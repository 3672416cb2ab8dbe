// dmip_tcl.cu — the fused score-training losses on tcgen05 (K2 DSM, K3 PINN / Score-FPE / DSM_PDE, the DPS passes).
//
// Same forward-mode jets as dmip_loss.cu (streams P | I | T | S_k | Q_ik per sample, SURVEY.md App. A.4/A.5), but every
// GEMM runs on the tensor cores.  Reference code replaced: losses.py:14-26,49-52,77-98,116-124,143-164,214-242,340-386
// and the loss.backward() of models/diffusion.py:100-102.
//
// Orientation ("transposed"): the WEIGHTS are the A operand (M = 128 output features per accumulator chunk), the 64 rows
// of a tile (sample x stream pairs) are the B operand (N = 64), so a TMEM lane is an output FEATURE and a thread that
// reads 32 accumulator columns holds ALL streams of its samples for that feature: the jet activation
// (phi, phi', phi'' coupling P -> T, S, Q) is thread-local — no shuffles, and tanh is evaluated once per sample and
// feature instead of once per stream.
// Precision: bf16x3 split product, a_hi w_hi + a_hi w_lo + a_lo w_hi, fp32 accumulation in tensor memory.
// Memory: the activations of one layer, hi and lo, are 64 rows x 512 features x 4 B = 128 KB of shared memory, as an
// MN-major 128B-swizzled B operand ([feature][row]: the epilogue thread of a feature writes 16-byte row chunks).  Every
// layer runs K-OUTER (all four 128-feature accumulator chunks are open, 4 x 64 TMEM columns, while the contraction
// walks the 64-feature K-blocks), so a layer's input is dead when its last MMA retires and the epilogue overwrites it
// IN PLACE with the next layer's input; the two TMEM halves alternate between consecutive layers, and the next layer's
// MMAs start as soon as its first K-blocks are written.
// Weight stream: hi / lo stages of 16 KB (128 features x 64 k, K-major, the sampler's stage format) in consumption
// order, bulk-TMA into a 5-slot ring.
// CTA pairs (kPair, the default): the two CTAs of a cluster issue ONE tcgen05.mma.cta_group::2 (M = 256, N = 128) over
// their two tiles; see the comment at kPair for what moves between the CTAs.
//
// Three kernels + pack:  k_tcl_fwd  (jets forward, per-sample loss terms, output adjoints, stashes for the backward),
//                        k_tcl_bwd  (adjoint rows P | I | T back through the layers, bias gradients),
//                        k_tcl_wgrad (dW_l = ADJ_l^T IN_l as split-K tcgen05 GEMMs over the stash images).
#include <stdlib.h>

#include "dmip_common.h"
#include "dmip_jets.cuh"
#include "dmip_ptx.cuh"
#include "dmip_tcl.h"

namespace dmip {

namespace {

constexpr int kNR = kTclRows;
constexpr int kWin = kTclWin;
constexpr int kStage = kTclStage;
constexpr int kSlots = 5;                 // weight ring: 5 x 16 KB
constexpr int kHHalf = 65536;             // 512 features x 64 rows x bf16 (hi OR lo)
constexpr int kInHalf = 8192;             // 64 features x 64 rows x bf16: operand of the first GEMM (hi OR lo)
constexpr int kThreads = 640;             // warps 0-15 row warps, 16 producer, 17 MMA issuer, 18-19 idle
constexpr int kRowThreads = 512;
constexpr int kNumRowWarps = 16;
constexpr int kProducerWarp = 16;
constexpr int kMmaWarp = 17;
constexpr int kCluster = 2;
constexpr int kRegsSmall = 32;
constexpr int kRegsRow = 112;
constexpr uint32_t kTmemCols = 512;       // two halves of 4 chunks x 64 columns (pair mode: 2 chunks x 128 columns)
// CTA-pair mode (default): the two CTAs of a cluster run ONE tcgen05.mma.cta_group::2 of M = 256, N = 128 per step instead
// of two M = 128, N = 64 instructions each.  An N = 64 shared-memory-operand instruction occupies the tensor pipe 32 of
// the ~96 cycles it takes (6 KB of operand reads); the pair instruction takes ~110 cycles for twice the work per SM.
// Every CTA keeps ITS 64-row tile as before (inputs, B operand in its own shared memory, stashes, loss stage); what is
// redistributed are the accumulators: CTA r holds the features of chunks r and r + 2 for the rows of BOTH tiles (128
// columns), so its epilogue threads write half of their output rows into the peer's shared memory — with st.async,
// whose completion bytes are counted on the peer's `rready` barrier: the writer neither fences nor arrives, the peer's
// receiver warp (18) forwards "rows landed" — and every "operand ready" barrier lives in the leader CTA (rank 0), which
// issues for the pair.  Each CTA streams only the weight stages of its own chunks (no multicast); the peer's MMA warp
// relays "stage landed" to the leader.
// -DDMIP_TCL_PAIR=0 builds the single-CTA kernels (cta_group::1, N = 64).
#ifndef DMIP_TCL_PAIR
#define DMIP_TCL_PAIR 1
#endif
constexpr bool kPair = DMIP_TCL_PAIR != 0;

constexpr int kOffHhi = 0;
constexpr int kOffHlo = kOffHhi + kHHalf;
constexpr int kOffIn = kOffHlo + kHHalf;                 // hi at +0, lo at +kInHalf
constexpr int kOffW = kOffIn + 2 * kInHalf;
constexpr int kOffBar = kOffW + kSlots * kStage;
constexpr int kNumBars = 2 * kSlots + 2 + 4 + 1 + kSlots + 1 + 4;
constexpr int kOffRed = kOffBar + ((kNumBars * 8 + 15) & ~15);   // float red[4], b3sum[64]
constexpr int kOffTmem = kOffRed + (4 + kTclSmallF) * 4;
constexpr int kSmemBytes = kOffTmem + 16;
static_assert(kSmemBytes <= 232448, "shared memory budget");

struct Bars {
  uint64_t* full;      // [kSlots]  weight stage landed (tx bytes)
  uint64_t* empty;     // [kSlots]  weight stage consumed (one tcgen05.commit per cluster CTA)
  uint64_t* acc_full;  // [2]       all MMAs of a layer complete (tcgen05.commit): TMEM half g & 1 is ready AND the layer's
                       //           shared-memory input is dead
  uint64_t* hready;    // [4]       K-blocks 2c, 2c+1 of the next B operand written (8 row warps each)
  uint64_t* in_ready;  // [1]       operand of the tile's first GEMM written (16 row warps)
  // pair mode: hready / in_ready are the LEADER's (arrivals from both CTAs: 16 row warps of the CTA that owns the chunk /
  // 32 row warps), and
  uint64_t* pfull;     // [kSlots]  leader: the peer's weight stage landed (relayed by the peer's MMA warp)
  uint64_t* xfree;     // [1]       the PEER's row warps have finished reading their staged outputs (forward loss stage):
                       //           its activation region may take the next tile's rows
  uint64_t* rready;    // [4]       this CTA's rows of chunk c, written by the PEER with st.async, have landed (32 KB of
                       //           transaction bytes per phase, armed and forwarded to hready[c] by the receiver warp)
};

__device__ __forceinline__ Bars make_bars(uint8_t* smem) {
  uint64_t* b = reinterpret_cast<uint64_t*>(smem + kOffBar);
  Bars B;
  B.full = b;
  B.empty = b + kSlots;
  B.acc_full = b + 2 * kSlots;
  B.hready = B.acc_full + 2;
  B.in_ready = B.hready + 4;
  B.pfull = B.in_ready + 1;
  B.xfree = B.pfull + kSlots;
  B.rready = B.xfree + 1;
  return B;
}

// see dmip_tc.cu: a value that went through a shuffle stays in a register instead of being re-loaded from the constant bank
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
template <int kRegs>
__device__ __forceinline__ void reg_dealloc() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegs)); }
template <int kRegs>
__device__ __forceinline__ void reg_alloc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegs)); }
// operand store of an epilogue thread: own shared memory, or (pair mode, rmbar != 0) an asynchronous store into the
// peer's shared memory whose arrival is counted on the peer's `rready` barrier — the writer neither fences nor arrives
__device__ __forceinline__ void st_operand_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d, uint32_t rmbar) {
  // (local rows take a plain st.shared on the CTA's own address: a st.shared::cluster on the mapa address of the own rank
  // is a GENERIC store — ST.E.128 behind an S2R SR_SWINHI per store, 6 % of the forward kernel's warp samples)
  if (kPair && rmbar != 0u) st_async_v4(addr, a, b, c, d, rmbar);
  else asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
constexpr uint32_t kRemoteChunkBytes = 8u * 32u * 8u * 16u;   // 8 warps x 32 features x (4 row chunks x hi, lo) x 16 B
// (a cluster-scope proxy fence would carry a GPU-scope membar that waits for every store of the thread in flight, global
// ones included: the first pair version spent 13 % of its warp samples there — rows of the peer's tile go by st.async)
__device__ __forceinline__ void fence_operand_stores() { fence_proxy_async_smem(); }
// arrival on a barrier of the leader CTA (pair mode: `leader_addr` = mapa of the barrier in CTA 0) or of this CTA
// — always with release at CLUSTER scope there: the stores it publishes may have gone to the peer's shared memory
__device__ __forceinline__ void arrive_issuer(uint64_t* bar, uint32_t leader_addr) {
  if (kPair) mbar_arrive_remote_relaxed(leader_addr);   // after fence_operand_stores(): its membar is the release
  else mbar_arrive(bar);
}
__device__ __forceinline__ void row_warps_sync() {   // named barrier over the 512 row-warp threads
  asm volatile("bar.sync 1, 512;" ::: "memory");
}

// ---- bf16 hi / lo split
__device__ __forceinline__ void split1(float x, unsigned short& hi, unsigned short& lo) {
  const uint32_t h = pack_bf16x2(x, 0.f) & 0xFFFFu;
  hi = static_cast<unsigned short>(h);
  lo = static_cast<unsigned short>(pack_bf16x2(x - __uint_as_float(h << 16), 0.f) & 0xFFFFu);
}
__device__ __forceinline__ void split2(float x0, float x1, uint32_t& hi, uint32_t& lo) {   // x0 in bits [0,16)
  hi = pack_bf16x2(x0, x1);
  lo = pack_bf16x2(x0 - __uint_as_float(hi << 16), x1 - __uint_as_float(hi & 0xFFFF0000u));
}
__device__ __forceinline__ float join1(unsigned short hi, unsigned short lo) {
  return __uint_as_float(static_cast<uint32_t>(hi) << 16) + __uint_as_float(static_cast<uint32_t>(lo) << 16);
}

// byte offset of (row, feature f) inside one 64-row block of a stash image with F features (dmip_tcl.h)
__device__ __forceinline__ uint32_t img_off(uint32_t row, uint32_t f) {
  return (f >> 6) * 8192u + (row >> 3) * 1024u + (row & 7u) * 128u + ((((f & 63u) >> 3) ^ (row & 7u)) << 4) + (f & 7u) * 2u;
}
// (feature k, row) of the MN-major B operand of a tile sits at byte (k / 8) * 1024 + (k % 8) * 128 + (((row / 8) ^ (k % 8)) << 4)
// + (row % 8) * 2: atoms of 1 KB = 8 k lines x 64 rows (the build_input functions and the epilogues write it that way)

// tanh to fp32 accuracy without the branch of tanhf: 1 - 2 / (e^{2|x|} + 1) on the two MUFU ops (ex2, rcp; absolute
// error ~3e-7, where the quotient cancels) and the odd Taylor polynomial below |x| = 0.04 (relative error < 1e-7 there).
// The epilogue of a layer's first accumulator chunks is on the path the next layer's MMAs wait for.
__device__ __forceinline__ float tanh_acc(float x) {
  const float ax = fabsf(x);
  float t;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(ax * 2.8853900817779268f));
  const float big = 1.0f - __fdividef(2.0f, t + 1.0f);
  const float x2 = x * x;
  const float small = ax * fmaf(x2, fmaf(x2, 0.13333333f, -0.33333334f), 1.0f);
  return copysignf(ax < 0.04f ? small : big, x);
}

// activation jets: value h, first and second derivative of phi at pre-activation z (layer 0: tanh(tanh), else tanh)
template <bool kFirst>
__device__ __forceinline__ void act_jet(float z, float& h, float& p1, float& p2) {
  if (kFirst) {
    const float u = tanh_acc(z);
    h = tanh_acc(u);
    const float du = 1.f - u * u;
    p1 = (1.f - h * h) * du;
    p2 = p1 * (-2.f * h * du - 2.f * u);
  } else {
    h = tanh_acc(z);
    p1 = 1.f - h * h;
    p2 = -2.f * h * p1;
  }
}

// stream set of a kernel instantiation (dmip_jets.cuh: the stream layout S)
template <int HAS_I, int HAS_T, int NT, int HAS_Q>
struct Cfg {
  static constexpr int kI = HAS_I, kT = HAS_T, kNT = NT, kQ = HAS_Q;
  static constexpr int NQ = HAS_Q ? NT * (NT + 1) / 2 : 0;
  static constexpr int NS = 1 + HAS_I + HAS_T + NT + NQ;   // streams per sample
  static constexpr int SPW = kWin / NS;                    // samples per 32-row window (forward)
  static constexpr int NADJ = 1 + HAS_I + HAS_T;           // adjoint streams per sample
  static constexpr int SPWB = kWin / NADJ;                 // samples per window (backward, stash blocks)
  static constexpr int sI = 1, sT = 1 + HAS_I, sS = sT + HAS_T, sQ = sS + NT;
  static_assert(NS <= kWin, "a sample's streams must fit one window");
};
// the stream set of the plain net's double backward (post == 5): P | T
template <class C>
constexpr bool kDoubleBwd = C::kT && !C::kI && C::kNT == 0;

// (block, row) of adjoint stream `a` of sample `smp` in the backward geometry
template <class C>
__device__ __forceinline__ void bwd_row(long long smp, int a, long long& block, uint32_t& row) {
  constexpr int kSpt = 2 * C::SPWB;
  block = smp / kSpt;
  const int rem = static_cast<int>(smp - block * kSpt);
  const int wb = rem / C::SPWB, jb = rem - wb * C::SPWB;
  row = static_cast<uint32_t>(wb * kWin + jb * C::NADJ + a);
}

// ---- timeline of CTA 0 (timing builds -DDMIP_JOBMARKS only; tools/tcl_timeline.py): four roles x [count, (clock << 16 | code)...]
#ifdef DMIP_JOBMARKS
__device__ unsigned long long* g_tcl_tl = nullptr;
__device__ int g_tcl_tl_cap = 0;
struct Tl {
  unsigned long long* p;
  unsigned int n, cap;
};
__device__ __forceinline__ Tl tl_open(int role, bool on) {
  Tl r = {nullptr, 0u, 0u};
  if (on && blockIdx.x == 0 && g_tcl_tl != nullptr) {
    const int seg = g_tcl_tl_cap / 4;
    r.p = g_tcl_tl + static_cast<size_t>(role) * seg;
    r.cap = static_cast<unsigned int>(seg - 1);
  }
  return r;
}
__device__ __forceinline__ void tl_mark(Tl& r, unsigned int code) {
  if (r.p != nullptr && r.n < r.cap) { r.p[1 + r.n] = (static_cast<unsigned long long>(clock64()) << 16) | code; ++r.n; }
}
__device__ __forceinline__ void tl_close(const Tl& r) { if (r.p != nullptr) r.p[0] = r.n; }
#define TL_OPEN(name, role, on) Tl name = tl_open(role, on)
#define TL_MARK(name, code) tl_mark(name, code)
#define TL_CLOSE(name) tl_close(name)
#else
#define TL_OPEN(name, role, on) ((void)0)
#define TL_MARK(name, code) ((void)0)
#define TL_CLOSE(name) ((void)0)
#endif

// ------------------------------------------------------------------------------------------------ producer / issuer
// Streams the n_stages weight stages of one tile pass, for every tile this CTA runs (whole warp, one elected lane issues).
// Single-CTA mode: both CTAs of the cluster walk the whole image, each fetches half of every stage and multicasts it.
// Pair mode: CTA r fetches, for every GEMM with four chunks, only the stages of ITS chunks r and r + 2 (image order: GEMM,
// K-block, chunk, hi | lo), and all stages of a one-chunk GEMM (both CTAs compute that chunk: each reads its own rows).
template <int kNG, int kLastChunks>
__device__ __forceinline__ void tcl_producer(const uint8_t* stages, int n_stages, int tile_first, int n_tiles, int tile_stride,
                                             uint8_t* sW, const Bars& B, uint32_t crank, uint16_t cmask) {
  int s = 0;
  uint32_t ph = 0;
  constexpr uint32_t part = kStage / kCluster;
  for (int tb = tile_first; tb < n_tiles; tb += tile_stride) {
    if (!kPair) {
      for (int st = 0; st < n_stages; ++st) {
        mbar_wait(&B.empty[s], ph ^ 1u, 0xA00 + s);   // slot released by the issuers of ALL cluster CTAs
        const uint8_t* g = stages + static_cast<size_t>(st) * kStage;
        if (elect_one()) {
          mbar_arrive_expect_tx(&B.full[s], kStage);
          if (kCluster == 1) bulk_g2s(sW + s * kStage, g, kStage, &B.full[s]);
          else bulk_g2s_multicast(sW + s * kStage + crank * part, g + crank * part, part, &B.full[s], cmask);
        }
        __syncwarp();
        if (++s == kSlots) { s = 0; ph ^= 1u; }
      }
    } else {
      int base = 0;   // first stage of GEMM g in the image
#pragma unroll 1
      for (int g = 0; g < kNG; ++g) {
        const int nkb = g == 0 ? 1 : 8;
        const int nc = g == kNG - 1 ? kLastChunks : 4;
        const int np = nc == 4 ? 2 : 1;
#pragma unroll 1
        for (int kb = 0; kb < nkb; ++kb)
#pragma unroll 1
          for (int p = 0; p < np; ++p)
#pragma unroll 1
            for (int hl = 0; hl < 2; ++hl) {
              const int c = nc == 4 ? static_cast<int>(crank) + 2 * p : 0;
              const int st = base + (kb * nc + c) * 2 + hl;
              mbar_wait(&B.empty[s], ph ^ 1u, 0xA00 + s);   // slot released by the leader's commit
              if (elect_one()) {
                mbar_arrive_expect_tx(&B.full[s], kStage);
                bulk_g2s(sW + s * kStage, stages + static_cast<size_t>(st) * kStage, kStage, &B.full[s]);
              }
              __syncwarp();
              if (++s == kSlots) { s = 0; ph ^= 1u; }
            }
        base += nkb * nc * 2;
      }
    }
  }
}

// Pair mode, MMA warp of the peer CTA (rank 1): tells the leader that a weight stage has landed in THIS CTA's ring.
__device__ __forceinline__ void tcl_relay(int n_stages_cta, int tile_first, int n_tiles, int tile_stride, const Bars& B) {
  int s = 0;
  uint32_t ph = 0;
  const uint32_t pfull0 = mapa_u32(&B.pfull[0], 0);
  for (int tb = tile_first; tb < n_tiles; tb += tile_stride) {
    for (int st = 0; st < n_stages_cta; ++st) {
      mbar_wait(&B.full[s], ph, 0xA80 + s);
      if (elect_one()) mbar_arrive_remote_relaxed(pfull0 + static_cast<uint32_t>(s) * 8u);
      __syncwarp();
      if (++s == kSlots) { s = 0; ph ^= 1u; }
    }
  }
}
// stages one CTA of a pair streams per tile
template <int kNG, int kLastChunks>
struct PairStages {
  static_assert(kNG >= 2, "a small-K GEMM followed by 512-deep ones");
  // GEMM 0: one K-block, two of its four chunks, hi | lo; the middle GEMMs: 8 K-blocks x 2 chunks x 2; the last GEMM:
  // 8 K-blocks x (2 of 4 chunks, or its only chunk) x 2
  static constexpr int value = 4 + (kNG - 2) * 32 + (kLastChunks == 4 ? 32 : 16);
};

// MMA issuer of one CTA: kNG GEMMs per tile; GEMM 0 reads the small operand (K = 16 k0steps), the others the 512-deep
// activations; all K-outer over 64-feature K-blocks with (up to) four open accumulator chunks; the last GEMM has
// kLastChunks chunks.  Per (K-block, chunk): the hi weight stage meets B hi and B lo, the lo stage meets B hi.
template <int kNG, int kLastChunks>
__device__ __forceinline__ void tcl_issuer(int k0steps, int tile_first, int n_tiles, int tile_stride, uint8_t* smem,
                                           uint32_t tmem_base, const Bars& B, uint16_t cmask) {
  int s = 0;
  uint32_t ph = 0, hr_par = 0, in_par = 0;
  uint32_t gc = 0;   // running GEMM counter: consecutive GEMMs alternate between the two TMEM halves, across tiles too
  const uint32_t in16 = (smem_u32(smem + kOffIn) & 0x3FFFFu) >> 4;
  const uint32_t h16 = (smem_u32(smem + kOffHhi) & 0x3FFFFu) >> 4;
  const uint32_t w16 = (smem_u32(smem + kOffW) & 0x3FFFFu) >> 4;
  const uint64_t descA = umma_smem_desc_sw128(0) & 0xFFFFFFFF00000000ull;           // K-major weights
  const uint64_t descB = umma_smem_desc(0, 1024, 1024);                             // MN-major rows: 8-k groups 1 KB apart
  constexpr uint32_t idesc = umma_idesc_bf16_major(128, kNR, 0, 1);
  for (int tb = tile_first; tb < n_tiles; tb += tile_stride) {
#pragma unroll 1
    for (int g = 0; g < kNG; ++g) {
      const int nkb = g == 0 ? 1 : 8;
      const int nc = g == kNG - 1 ? kLastChunks : 4;
      const int nk16 = g == 0 ? k0steps : 4;
      const uint32_t b_base = g == 0 ? in16 : h16;
      const uint32_t b_half = (g == 0 ? kInHalf : kHHalf) >> 4;
      const uint32_t set = gc & 1u;
      ++gc;
      const uint32_t acc0 = tmem_base + set * 256u;
#pragma unroll 1
      for (int kb = 0; kb < nkb; ++kb) {
        if (g == 0) {
          mbar_wait(B.in_ready, in_par, 0xB00);
          in_par ^= 1u;
        } else if ((kb & 1) == 0) {
          const int c = kb >> 1;
          mbar_wait(&B.hready[c], (hr_par >> c) & 1u, 0xB10 + c);
          hr_par ^= 1u << c;
        }
        tc_fence_after();
        const uint32_t b16 = b_base + static_cast<uint32_t>(kb) * 512u;   // 8 k-groups x 1 KB per K-block
#pragma unroll 1
        for (int c = 0; c < nc; ++c) {
          const uint32_t d = acc0 + static_cast<uint32_t>(c) * kNR;
          // hi stage x (B hi, B lo)
          mbar_wait(&B.full[s], ph, 0xB20 + s);
          tc_fence_after();
          uint32_t a16 = w16 + static_cast<uint32_t>(s) * (kStage >> 4);
          if (elect_one()) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (j < nk16) {
                umma_ss(d, descA | (a16 + j * 2), descB | (b16 + j * 128), idesc, (kb | j) != 0 ? 1u : 0u);
                umma_ss(d, descA | (a16 + j * 2), descB | (b16 + b_half + j * 128), idesc, 1u);
              }
            tc_commit_multicast(&B.empty[s], cmask);
          }
          __syncwarp();
          if (++s == kSlots) { s = 0; ph ^= 1u; }
          // lo stage x B hi
          mbar_wait(&B.full[s], ph, 0xB30 + s);
          tc_fence_after();
          a16 = w16 + static_cast<uint32_t>(s) * (kStage >> 4);
          if (elect_one()) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (j < nk16) umma_ss(d, descA | (a16 + j * 2), descB | (b16 + j * 128), idesc, 1u);
            tc_commit_multicast(&B.empty[s], cmask);
            if (kb == nkb - 1 && c == nc - 1) tc_commit(&B.acc_full[set]);
          }
          __syncwarp();
          if (++s == kSlots) { s = 0; ph ^= 1u; }
        }
      }
    }
  }
}

// MMA issuer of the LEADER CTA in pair mode: the same GEMM sequence with tcgen05.mma.cta_group::2 — M = 256 (chunk r + 2p
// from CTA r's ring slot), N = 128 (64 rows from each CTA's operand region, same CTA-relative address), accumulator p at
// columns p * 128 of the TMEM half in both CTAs.  A one-chunk GEMM runs with the same stage in both rings: each CTA ends
// up with that chunk for all 128 rows and reads its own 64.  Every commit is multicast to both CTAs.
template <int kNG, int kLastChunks>
__device__ __forceinline__ void tcl_issuer_pair(int k0steps, int tile_first, int n_tiles, int tile_stride, uint8_t* smem,
                                                uint32_t tmem_base, const Bars& B) {
  int s = 0;
  uint32_t ph = 0, hr_par = 0, in_par = 0;
  uint32_t gc = 0;
  const uint32_t in16 = (smem_u32(smem + kOffIn) & 0x3FFFFu) >> 4;
  const uint32_t h16 = (smem_u32(smem + kOffHhi) & 0x3FFFFu) >> 4;
  const uint32_t w16 = (smem_u32(smem + kOffW) & 0x3FFFFu) >> 4;
  const uint64_t descA = umma_smem_desc_sw128(0) & 0xFFFFFFFF00000000ull;
  const uint64_t descB = umma_smem_desc(0, 1024, 1024);
  constexpr uint32_t idesc = umma_idesc_bf16_major(256, 2 * kNR, 0, 1);
  constexpr uint16_t both = 0x3;
  TL_OPEN(tl, 0, (threadIdx.x & 31) == 0 && kNG == 4);   // the forward pass (the backward pass of a loss has three GEMMs)
  for (int tb = tile_first; tb < n_tiles; tb += tile_stride) {
#pragma unroll 1
    for (int g = 0; g < kNG; ++g) {
      TL_MARK(tl, 0x100u | g);
      const int nkb = g == 0 ? 1 : 8;
      const int np = (g == kNG - 1 ? kLastChunks : 4) == 4 ? 2 : 1;
      const int nk16 = g == 0 ? k0steps : 4;
      const uint32_t b_base = g == 0 ? in16 : h16;
      const uint32_t b_half = (g == 0 ? kInHalf : kHHalf) >> 4;
      const uint32_t set = gc & 1u;
      ++gc;
      const uint32_t acc0 = tmem_base + set * 256u;
#pragma unroll 1
      for (int kb = 0; kb < nkb; ++kb) {
        if (g == 0) {
          mbar_wait_cluster(B.in_ready, in_par, 0xB00);
          in_par ^= 1u;
        } else if ((kb & 1) == 0) {
          const int c = kb >> 1;
          mbar_wait_cluster(&B.hready[c], (hr_par >> c) & 1u, 0xB10 + c);
          hr_par ^= 1u << c;
          TL_MARK(tl, 0x200u | (g << 4) | c);
        }
        tc_fence_after();
        const uint32_t b16 = b_base + static_cast<uint32_t>(kb) * 512u;
#pragma unroll 1
        for (int p = 0; p < np; ++p) {
          const uint32_t d = acc0 + static_cast<uint32_t>(p) * (2 * kNR);
          // hi stage x (B hi, B lo)
          mbar_wait(&B.full[s], ph, 0xB20 + s);
          mbar_wait_cluster(&B.pfull[s], ph, 0xB40 + s);
          tc_fence_after();
          uint32_t a16 = w16 + static_cast<uint32_t>(s) * (kStage >> 4);
          if (elect_one()) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (j < nk16) {
                umma_ss_pair(d, descA | (a16 + j * 2), descB | (b16 + j * 128), idesc, (kb | j) != 0 ? 1u : 0u);
                umma_ss_pair(d, descA | (a16 + j * 2), descB | (b16 + b_half + j * 128), idesc, 1u);
              }
            tc_commit_pair(&B.empty[s], both);
          }
          __syncwarp();
          if (++s == kSlots) { s = 0; ph ^= 1u; }
          // lo stage x B hi
          mbar_wait(&B.full[s], ph, 0xB30 + s);
          mbar_wait_cluster(&B.pfull[s], ph, 0xB50 + s);
          tc_fence_after();
          a16 = w16 + static_cast<uint32_t>(s) * (kStage >> 4);
          if (elect_one()) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (j < nk16) umma_ss_pair(d, descA | (a16 + j * 2), descB | (b16 + j * 128), idesc, 1u);
            tc_commit_pair(&B.empty[s], both);
            if (kb == nkb - 1 && p == np - 1) tc_commit_pair(&B.acc_full[set], both);
          }
          __syncwarp();
          if (++s == kSlots) { s = 0; ph ^= 1u; }
        }
      }
      TL_MARK(tl, 0x300u | g);
    }
  }
  TL_CLOSE(tl);
}

// Pair mode, warp 18 of each CTA: per layer that produces an operand, and per chunk owned by the PEER, arm this CTA's rready
// barrier with the bytes the peer's st.async stores will deliver, wait for them, make them visible to the tensor core
// and tell the leader's issuer (hready[c]).
constexpr int kReceiverWarp = 18;
__device__ __forceinline__ void tcl_receiver(int n_operand_layers, int tile_first, int n_tiles, int tile_stride, const Bars& B,
                                             uint32_t crank) {
  uint32_t par = 0;
  const uint32_t hready_leader = mapa_u32(&B.hready[0], 0);
  for (int tb = tile_first; tb < n_tiles; tb += tile_stride)
    for (int l = 0; l < n_operand_layers; ++l)
      for (int ci = 0; ci < 2; ++ci) {
        const uint32_t c = (1u - crank) + 2u * static_cast<uint32_t>(ci);
        if (elect_one()) mbar_arrive_expect_tx(&B.rready[c], kRemoteChunkBytes);
        __syncwarp();
        mbar_wait_cluster(&B.rready[c], (par >> c) & 1u, 0xA90 + c);
        par ^= 1u << c;
        fence_proxy_async_smem();
        if (elect_one()) mbar_arrive_remote_relaxed(hready_leader + c * 8u);
        __syncwarp();
      }
}

// the three service roles of the warps above the row warps
template <int kNG, int kLastChunks>
__device__ __forceinline__ void tcl_service_warps(int warp, const uint8_t* stages, int n_stages, int k0steps, int tile_first,
                                                  int n_tiles, int tile_stride, uint8_t* smem, uint32_t tmem_base,
                                                  const Bars& B, uint32_t crank, uint16_t cmask) {
  if (warp == kProducerWarp) {
    tcl_producer<kNG, kLastChunks>(stages, n_stages, tile_first, n_tiles, tile_stride, smem + kOffW, B, crank, cmask);
  } else if (warp == kMmaWarp) {
    if (!kPair) tcl_issuer<kNG, kLastChunks>(k0steps, tile_first, n_tiles, tile_stride, smem, tmem_base, B, cmask);
    else if (crank == 0u) tcl_issuer_pair<kNG, kLastChunks>(k0steps, tile_first, n_tiles, tile_stride, smem, tmem_base, B);
    else tcl_relay(PairStages<kNG, kLastChunks>::value, tile_first, n_tiles, tile_stride, B);
  } else if (kPair && warp == kReceiverWarp) {
    // every GEMM but the last is followed by an epilogue that writes the next operand
    tcl_receiver(kNG - 1, tile_first, n_tiles, tile_stride, B, crank);
  }
}

// one-time setup shared by both kernels; returns tmem_base
__device__ __forceinline__ uint32_t tcl_setup(uint8_t* smem, const Bars& B, int warp, int lane) {
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(smem + kOffTmem);
  if ((smem_u32(smem) & 1023u) != 0u) __trap();
  if (warp == kProducerWarp && lane == 0) {
    for (int i = 0; i < kSlots; ++i) {
      mbar_init(&B.full[i], 1);
      mbar_init(&B.empty[i], kPair ? 1u : static_cast<uint32_t>(kCluster));   // pair mode: the leader's commit only
      mbar_init(&B.pfull[i], 1);
    }
    mbar_init(&B.acc_full[0], 1);
    mbar_init(&B.acc_full[1], 1);
    // single-CTA: 4 lane quarters x 2 windows; pair: all 16 row warps of the CTA that owns the chunk
    // (pair: the 8 warps of the chunk's owner whose rows are local + the receiver warp of the CTA that got the other rows)
    for (int i = 0; i < 4; ++i) mbar_init(&B.hready[i], kPair ? 9 : 8);
    for (int i = 0; i < 4; ++i) mbar_init(&B.rready[i], 1);
    mbar_init(B.in_ready, kPair ? 2 * kNumRowWarps : kNumRowWarps);
    mbar_init(B.xfree, kNumRowWarps);
    fence_barrier_init();
  }
  if (!kPair && warp == kMmaWarp) tmem_alloc<kTmemCols>(tmem_holder);
  // the operand regions must hold finite values from the start (zero rows / zero K padding meet zero weights)
  for (int i = threadIdx.x; i < kOffW / 16; i += kThreads) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
  float* red = reinterpret_cast<float*>(smem + kOffRed);
  for (int i = threadIdx.x; i < 4 + kTclSmallF; i += kThreads) red[i] = 0.f;
  fence_proxy_async_smem();
  if (kPair) {
    // both CTAs exist and their mbarriers are initialised before the pair allocation (one warp in EACH CTA)
    cluster_sync_all();
    if (warp == kMmaWarp) tmem_alloc_pair<kTmemCols>(tmem_holder);
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    return __shfl_sync(0xffffffffu, *tmem_holder, 0);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_holder, 0);
  if (kCluster > 1) cluster_sync_all();   // every CTA's mbarriers exist before any multicast / remote commit
  return tmem_base;
}

__device__ __forceinline__ void tcl_teardown(uint32_t tmem_base, int warp) {
  tc_fence_before();
  __syncthreads();
  if (kCluster > 1) cluster_sync_all();
  if (warp == kMmaWarp) {
    tc_fence_after();
    if (kPair) tmem_dealloc_pair<kTmemCols>(tmem_base);
    else tmem_dealloc<kTmemCols>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------ forward
// Layer-0 operand of tile `tile`: rows (sample, stream) x input columns, written as the MN-major B operand of GEMM 0
// and — for the adjoint streams P | I | T — into the IN_0 stash the weight-gradient GEMM reads.  Thread mapping: lanes
// walk the input columns (coalesced stash rows), warps walk the rows.
template <class C>
__device__ __forceinline__ void fwd_build_input(const TclDev& P, long long tile, bool tile_ok, uint8_t* sIn, int t) {
  // One row x 8 consecutive input columns per thread (512 threads = 64 rows x 8 column groups): the per-sample terms
  // (two expf, a sqrt, the loads of t / x / y / eps) are evaluated once per row, only the warps of a column group below
  // in_dim do any arithmetic, and a stash row is two 16-byte stores.  (One column x 8 rows per thread — the first version —
  // left the five lanes with k < in_dim walking 8 rows of dependent loads serially: 15 K cycles per tile on the warps the
  // next layer's epilogue was waiting for, tools/tcl_timeline.py.)
  const int row = t & 63, kg = t >> 6;
  const int w = row >> 5, rw = row & 31;
  const int j = rw / C::NS, st = rw - j * C::NS;
  const long long smp = tile * (2 * C::SPW) + w * C::SPW + j;
  const bool live_row = tile_ok && j < C::SPW && smp < P.B;
  float v[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) v[e] = 0.f;
  if (live_row && kg * 8 < P.in_dim) {
    if (kDoubleBwd<C> && P.post == 5 && st == C::sT) {
      // double backward: the T rows carry the caller's tangent direction v
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int k = kg * 8 + e;
        if (k < P.in_dim) v[e] = P.dir[smp * P.in_dim + k];
      }
    } else if (P.post == 4 || (kDoubleBwd<C> && P.post == 5)) {
      // plain net forward (and the P rows of its double backward): cat[x, cond, t] as given (nets.py:32-35, :52-57)
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int k = kg * 8 + e;
        if (k < P.xdim) v[e] = P.x[smp * P.xdim + k];
        else if (k < P.xdim + P.ydim) v[e] = P.y[smp * P.ydim + (k - P.xdim)];
        else if (k < P.in_dim) v[e] = P.t[smp];
      }
    } else {
      const SampleSde vp = sample_sde(P, smp);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int k = kg * 8 + e;
        if (k < P.in_dim) v[e] = jet_input(P, C{}, vp, smp, st, k);
      }
    }
  }
  uint32_t hi[4], lo[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) split2(v[2 * e], v[2 * e + 1], hi[e], lo[e]);
  // MN-major B operand: column k = kg * 8 + e is line e of atom kg; this row's element sits in chunk (row / 8) ^ e
  uint8_t* atom = sIn + kg * 1024 + (row & 7) * 2;
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    uint8_t* q = atom + e * 128 + (((row >> 3) ^ e) << 4);
    const uint32_t h2 = hi[e >> 1], l2 = lo[e >> 1];
    *reinterpret_cast<unsigned short*>(q) = static_cast<unsigned short>((e & 1) ? (h2 >> 16) : (h2 & 0xFFFFu));
    *reinterpret_cast<unsigned short*>(q + kInHalf) = static_cast<unsigned short>((e & 1) ? (l2 >> 16) : (l2 & 0xFFFFu));
  }
  // inputs of layer 0 for the adjoint streams (weight-gradient operand), in the backward geometry: 8 features = 16 bytes
  const int a = (st == 0) ? 0 : (C::kI && st == C::sI) ? 1 : (C::kT && st == C::sT) ? (1 + C::kI) : -1;
  if (live_row && a >= 0) {
    long long blk;
    uint32_t rb;
    bwd_row<C>(smp, a, blk, rb);
    const size_t o = static_cast<size_t>(blk) * (kTclSmallF * 128) + img_off(rb, static_cast<uint32_t>(kg * 8));
    *reinterpret_cast<uint4*>(P.in_img[0][0] + o) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(P.in_img[0][1] + o) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}

// One (layer, chunk, window) item of the forward epilogue: thread = feature n of the layer's output.
template <class C, bool kFirst>
__device__ __forceinline__ void fwd_item(const TclDev& P, int g, uint32_t taddr, int n, float bias, long long smp0,
                                         bool tile_ok, int w, uint32_t hdst, uint32_t rmbar, uint32_t (&v)[32]) {
  tmem_ld32(taddr, v);
  tc_wait_ld();
  const bool full = tile_ok && smp0 + C::SPW <= P.B;     // warp-uniform
  float* sst0 = P.st[g] + (smp0 * C::NADJ) * 512 + n;
#pragma unroll
  for (int j = 0; j < C::SPW; ++j) {
    const int base = j * C::NS;
    float h, p1, p2;
    act_jet<kFirst>(__uint_as_float(v[base]) + bias, h, p1, p2);
    v[base] = __float_as_uint(h);
    float hI = 0.f, q1 = 0.f, hdT = 0.f, cT = 0.f;
    if (C::kI) {
      float q2;
      act_jet<kFirst>(__uint_as_float(v[base + C::sI]) + bias, hI, q1, q2);
      v[base + C::sI] = __float_as_uint(hI);
    }
    if (C::kT) {
      const float zd = __uint_as_float(v[base + C::sT]);
      hdT = p1 * zd;
      cT = p2 * zd;
      v[base + C::sT] = __float_as_uint(hdT);
    }
    if (C::kNT > 0) {
      float zs[C::kNT > 0 ? C::kNT : 1];
#pragma unroll
      for (int k = 0; k < C::kNT; ++k) zs[k] = __uint_as_float(v[base + C::sS + k]);
      if (C::kQ) {
#pragma unroll
        for (int i = 0; i < C::kNT; ++i)
#pragma unroll
          for (int k = i; k < C::kNT; ++k) {
            const int q = base + C::sQ + q_index(i, k, C::kNT);
            v[q] = __float_as_uint(fmaf(p1, __uint_as_float(v[q]), p2 * zs[i] * zs[k]));
          }
      }
#pragma unroll
      for (int k = 0; k < C::kNT; ++k) v[base + C::sS + k] = __float_as_uint(p1 * zs[k]);
    }
    // derivative state the backward epilogue needs (fp32, coalesced; dmip_tcl.h: st).  Offsets from one base pointer
    // are compile-time constants; a window that lies inside the batch (all but the last tile) stores unpredicated.
    // Pair mode, layers 1 and 2: stored by fwd_state_from_outputs AFTER the operand fence instead.
    if ((!kPair || kFirst) && (full || (tile_ok && smp0 + j < P.B))) {
      float* sst = sst0 + static_cast<size_t>(j) * (C::NADJ * 512);
      sst[0] = p1;
      if (C::kI) sst[512] = q1;
      if (C::kT) sst[(1 + C::kI) * 512] = cT;
    }
  }
#pragma unroll
  for (int r = C::SPW * C::NS; r < kWin; ++r) v[r] = 0u;   // padding rows of the window
  // next layer's B operand: feature n, rows w*32 .. w*32+31 = four 16-byte chunks, hi and lo (hdst: the hi activation
  // region of the CTA that owns the rows — this CTA, or in pair mode either one)
  const uint32_t hrow = hdst + (static_cast<uint32_t>(n) >> 3) * 1024u + (static_cast<uint32_t>(n) & 7u) * 128u;
  const uint32_t line = static_cast<uint32_t>(n) & 7u;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int e = 0; e < 4; ++e)
      split2(__uint_as_float(v[i * 8 + 2 * e]), __uint_as_float(v[i * 8 + 2 * e + 1]), hi[e], lo[e]);
    const uint32_t co = ((static_cast<uint32_t>(w * 4 + i) ^ line) << 4);
    st_operand_v4(hrow + co, hi[0], hi[1], hi[2], hi[3], rmbar);
    st_operand_v4(hrow + kHHalf + co, lo[0], lo[1], lo[2], lo[3], rmbar);
  }
}

// Pair mode, tanh layers: the derivative state of fwd_item from the layer's OUTPUTS still in v[] (h, h_I, p1 zd_T):
//   phi'(z_P) = 1 - h^2,  phi'(z_I) = 1 - h_I^2,  phi''(z_P) zd_T = -2 h (p1 zd_T)  — after the next layer's MMAs were
// released, so that the operand fence does not wait for these global stores.
template <class C>
__device__ __forceinline__ void fwd_state_from_outputs(const TclDev& P, int g, int n, long long smp0, bool tile_ok,
                                                       const uint32_t (&v)[32]) {
  const bool full = tile_ok && smp0 + C::SPW <= P.B;
  float* sst0 = P.st[g] + (smp0 * C::NADJ) * 512 + n;
#pragma unroll
  for (int j = 0; j < C::SPW; ++j) {
    if (full || (tile_ok && smp0 + j < P.B)) {
      const int base = j * C::NS;
      float* sst = sst0 + static_cast<size_t>(j) * (C::NADJ * 512);
      const float h = __uint_as_float(v[base]);
      sst[0] = 1.f - h * h;
      if (C::kI) { const float hI = __uint_as_float(v[base + C::sI]); sst[512] = 1.f - hI * hI; }
      if (C::kT) sst[(1 + C::kI) * 512] = -2.f * h * __uint_as_float(v[base + C::sT]);
    }
  }
}

// Second half of an item, AFTER the next layer's MMAs were told the K-blocks are there: the outputs of the adjoint streams
// P | I | T (still in v[]) go to the IN_{g+1} stash image (bf16 hi/lo, backward geometry: weight-gradient operand).
template <class C>
__device__ __forceinline__ void fwd_stash(const TclDev& P, int g, int n, long long tile, long long smp0, bool tile_ok, int w,
                                          const uint32_t (&v)[32]) {
  const uint32_t nterm = (static_cast<uint32_t>(n) >> 6) * 8192u + (static_cast<uint32_t>(n) & 7u) * 2u;
  const uint32_t nchunk = (static_cast<uint32_t>(n) & 63u) >> 3;
  if (C::NS == C::NADJ) {
    // every stream is an adjoint stream (DSM, cScoreFPE, adjoint-route passes): the forward tile IS the stash block and
    // window row r is block row w*32 + r — all offsets but the swizzle term are compile-time constants
    if (!tile_ok) return;
    uint8_t* ihi = P.in_img[g + 1][0] + static_cast<size_t>(tile) * (512 * 128) + nterm + static_cast<uint32_t>(w) * 4096u;
    uint8_t* ilo = P.in_img[g + 1][1] + static_cast<size_t>(tile) * (512 * 128) + nterm + static_cast<uint32_t>(w) * 4096u;
    const uint32_t nc4 = nchunk << 4;                  // swizzle term: one XOR with an immediate per row
    const bool full = smp0 + C::SPW <= P.B;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const uint32_t xo = i * 128u + (nc4 ^ (static_cast<uint32_t>(i) << 4));
#pragma unroll
      for (int q = 0; q < kWin / 8; ++q) {
        const int r = q * 8 + i;
        if (r < C::SPW * C::NS && (full || smp0 + r / C::NS < P.B)) {
          unsigned short hi, lo;
          split1(__uint_as_float(v[r]), hi, lo);
          *reinterpret_cast<unsigned short*>(ihi + q * 1024u + xo) = hi;
          *reinterpret_cast<unsigned short*>(ilo + q * 1024u + xo) = lo;
        }
      }
    }
    return;
  }
#pragma unroll
  for (int j = 0; j < C::SPW; ++j) {
    const long long smp = smp0 + j;
    if (tile_ok && smp < P.B) {
      long long blk;
      uint32_t rb;
      bwd_row<C>(smp, 0, blk, rb);
      uint8_t* ihi = P.in_img[g + 1][0] + static_cast<size_t>(blk) * (512 * 128) + nterm;
      uint8_t* ilo = P.in_img[g + 1][1] + static_cast<size_t>(blk) * (512 * 128) + nterm;
#pragma unroll
      for (int a = 0; a < C::NADJ; ++a) {
        const int st = a == 0 ? 0 : (C::kI && a == 1) ? C::sI : C::sT;
        const uint32_t r2 = rb + a;
        const uint32_t o = (r2 >> 3) * 1024u + (r2 & 7u) * 128u + ((nchunk ^ (r2 & 7u)) << 4);
        unsigned short hi, lo;
        split1(__uint_as_float(v[j * C::NS + st]), hi, lo);
        *reinterpret_cast<unsigned short*>(ihi + o) = hi;
        *reinterpret_cast<unsigned short*>(ilo + o) = lo;
      }
    }
  }
}

// staged net outputs of one sample: o[stream * od + component], bias already added to the primal rows
struct TclOuts {
  const float* o;
  int od;
  __device__ __forceinline__ float primal(int s, int c) const { return o[s * od + c]; }
  __device__ __forceinline__ float tangent(int s, int c) const { return o[s * od + c]; }
};

// Per-sample loss terms and output adjoints from the staged net outputs (all streams of the tile's samples):
// dmip_jets.cuh, jet_loss_item.
template <class C>
__device__ __forceinline__ void fwd_loss_stage(const TclDev& P, long long s0, bool tile_ok, const float* outs, float* red,
                                               float* b3sum, int t) {
  constexpr int spt = 2 * C::SPW;
  const int od = P.out_dim;
  const int n_items = spt * od;
  for (int base = 0; base < n_items; base += kRowThreads) {
    const int idx = base + t;
    const int sl = idx / od, j = idx - sl * od;
    const long long smp = s0 + sl;
    float l_dsm = 0.f, l_ic = 0.f, l_pde = 0.f;
    if (idx < n_items && tile_ok && smp < P.B) {
      const int row0 = (sl / C::SPW) * kWin + (sl % C::SPW) * C::NS;
      if (P.post == 4) {
        // plain net forward (dmip_mlp_forward_stash): the staged outputs are the result
        P.net_out[smp * od + j] = outs[row0 * od + j];
      } else if (kDoubleBwd<C> && P.post == 5) {
        // double backward: the T output J v is a result; the backward reverses u^T J v (output adjoints P: 0, T: u), and
        // nothing reaches the output bias
        if (P.net_out != nullptr) P.net_out[smp * od + j] = outs[(row0 + C::sT) * od + j];
        P.abar[(smp * C::NADJ) * od + j] = 0.f;
        P.abar[(smp * C::NADJ + C::sT) * od + j] = P.grad_out[smp * od + j];
      } else {
        const float gb = jet_loss_item(P, C{}, TclOuts{outs + row0 * od, od}, P.abar, od, smp, j, l_dsm, l_ic, l_pde);
        atomicAdd(&b3sum[j], gb);                    // d loss / d b3[j]: the primal rows P and I
      }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      l_dsm += __shfl_xor_sync(0xffffffffu, l_dsm, off);
      l_ic += __shfl_xor_sync(0xffffffffu, l_ic, off);
      l_pde += __shfl_xor_sync(0xffffffffu, l_pde, off);
    }
    if ((t & 31) == 0) {
      atomicAdd(&red[1], l_dsm);
      atomicAdd(&red[2], l_ic);
      atomicAdd(&red[3], l_pde);
    }
  }
}

template <class C>
__global__ void __launch_bounds__(kThreads, 1) k_tcl_fwd(const __grid_constant__ TclDev P) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const Bars B = make_bars(smem);
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const uint32_t tmem_base = tcl_setup(smem, B, warp, lane);
  const uint32_t crank = kCluster > 1 ? cluster_ctarank() : 0u;
  const uint16_t cmask = static_cast<uint16_t>((1u << kCluster) - 1u);
  const int n_tiles = keep(static_cast<int>(P.n_tiles_fwd));
  const int tile_first = static_cast<int>(blockIdx.x / kCluster) * kCluster;
  const int tile_stride = keep(static_cast<int>(gridDim.x));

  if (warp >= kNumRowWarps) {
    reg_dealloc<kRegsSmall>();
    tcl_service_warps<4, 1>(warp, keep(P.stages_fwd), kTclFwdStages, keep(P.k0steps_fwd), tile_first, n_tiles, tile_stride,
                            smem, tmem_base, B, crank, cmask);
  } else {
    reg_alloc<kRegsRow>();
    const int q = warp & 3, cgp = warp >> 2;
    // single-CTA: this warp's window w of the CTA's tile; its chunks are c_first and c_first + 2.
    // pair: the CTA's chunks are crank and crank + 2; the warp takes window w of the tile of CTA `tsel` (columns
    // tsel * 64 + w * 32 of the 128-column accumulators).
    const int w = cgp & 1;
    const int c_first = kPair ? static_cast<int>(crank) : cgp >> 1;
    const int tsel = kPair ? cgp >> 1 : static_cast<int>(crank);
    const int t = threadIdx.x;
    const uint32_t lane_taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const uint32_t hdst = (kPair && tsel != static_cast<int>(crank)) ? mapa_u32(smem + kOffHhi, static_cast<uint32_t>(tsel))
                                                                      : smem_u32(smem + kOffHhi);
    const uint32_t in_ready_leader = kPair ? mapa_u32(B.in_ready, 0) : 0u;
    const uint32_t hready_leader = kPair ? mapa_u32(&B.hready[0], 0) : 0u;
    const uint32_t xfree_peer = kPair ? mapa_u32(B.xfree, crank ^ 1u) : 0u;
    const bool remote = kPair && tsel != static_cast<int>(crank);       // this warp's rows live in the peer's shared memory
    const uint32_t rready_dst = remote ? mapa_u32(&B.rready[0], static_cast<uint32_t>(tsel)) : 0u;
    uint32_t xpar = 0;
    TL_OPEN(tl, warp == 0 ? 1 : warp == 8 ? 2 : 3, lane == 0 && (warp == 0 || warp == 8 || warp == 15));
    float* red = reinterpret_cast<float*>(smem + kOffRed);
    float* b3sum = red + 4;
    float* outs = reinterpret_cast<float*>(smem + kOffHhi);
    uint32_t par0 = 0, par1 = 0;                        // phases of acc_full[0], acc_full[1]
    float bias[3][2];                                   // this thread's two features per hidden layer (an L2 round trip
#pragma unroll                                          // per item otherwise, on the path the next layer's MMAs wait for)
    for (int g = 0; g < 3; ++g)
#pragma unroll
      for (int ci = 0; ci < 2; ++ci) bias[g][ci] = __ldg(P.b[g] + (c_first + 2 * ci) * 128 + q * 32 + lane);
    {
      const bool ok = tile_first + static_cast<int>(crank) < n_tiles;
      fwd_build_input<C>(P, tile_first + static_cast<int>(crank), ok, smem + kOffIn, t);
      fence_operand_stores();
      __syncwarp();
      if (lane == 0) arrive_issuer(B.in_ready, in_ready_leader);
    }
    for (int tb = tile_first; tb < n_tiles; tb += tile_stride) {
      const bool tile_ok = tb + static_cast<int>(crank) < n_tiles;      // this CTA's own tile (inputs, loss stage)
      const long long tile = tb + static_cast<int>(crank);
      const long long s0 = tile * (2 * C::SPW);
      const long long etile = tb + tsel;                                // the tile whose rows this warp's items hold
      const bool etile_ok = etile < n_tiles;
      const long long smp0 = etile * (2 * C::SPW) + w * C::SPW;
#pragma unroll 1
      for (int g = 0; g < 3; ++g) {
        if (g & 1) { mbar_wait(&B.acc_full[1], par1, 0xC01); par1 ^= 1u; }
        else { mbar_wait(&B.acc_full[0], par0, 0xC00); par0 ^= 1u; }
        tc_fence_after();
        TL_MARK(tl, 0x400u | g);
        if (kPair && g == 0 && tb != tile_first && tsel != static_cast<int>(crank)) {
          // the peer's activation region still holds its staged outputs of the previous tile until its loss stage is done
          mbar_wait_cluster(B.xfree, xpar, 0xC10);
          xpar ^= 1u;
        }
#pragma unroll 1
        for (int ci = 0; ci < 2; ++ci) {
          const int c = c_first + 2 * ci;
          const int n = c * 128 + q * 32 + lane;
          const uint32_t taddr = lane_taddr + static_cast<uint32_t>((g & 1) * 256) +
                                 (kPair ? static_cast<uint32_t>(ci * 2 * kNR + tsel * kNR + w * kWin)
                                        : static_cast<uint32_t>(c * kNR + w * kWin));
          // register select (the loops stay rolled: six copies of the item body would not fit the instruction cache)
          const float bs = g == 0 ? (ci ? bias[0][1] : bias[0][0]) : g == 1 ? (ci ? bias[1][1] : bias[1][0]) : (ci ? bias[2][1] : bias[2][0]);
          uint32_t v[32];
          const uint32_t rmbar = remote ? rready_dst + static_cast<uint32_t>(c) * 8u : 0u;
          if (g == 0) fwd_item<C, true>(P, g, taddr, n, bs, smp0, etile_ok, w, hdst, rmbar, v);
          else fwd_item<C, false>(P, g, taddr, n, bs, smp0, etile_ok, w, hdst, rmbar, v);
          if (!remote) {   // remote rows: the peer's receiver warp sees them land (rready) and tells the issuer
            fence_operand_stores();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) arrive_issuer(&B.hready[c], hready_leader + static_cast<uint32_t>(c) * 8u);
          }
          TL_MARK(tl, 0x500u | (g << 4) | ci);
          if (kPair && g != 0) fwd_state_from_outputs<C>(P, g, n, smp0, etile_ok, v);
          fwd_stash<C>(P, g, n, etile, smp0, etile_ok, w, v);
          TL_MARK(tl, 0x600u | (g << 4) | ci);
        }
        if (g == 1 && tb + tile_stride < n_tiles) {
          // GEMM 0 of this tile has retired (acc_full[0] above): the small operand region takes the next tile's inputs
          const int nt = tb + tile_stride + static_cast<int>(crank);
          fwd_build_input<C>(P, nt, nt < n_tiles, smem + kOffIn, t);
          fence_operand_stores();
          __syncwarp();
          if (lane == 0) arrive_issuer(B.in_ready, in_ready_leader);
        }
      }
      // ---- output layer: accumulator chunk 0 of TMEM half 1 -> staged outputs (the activation region is dead now).
      // Pair mode: both CTAs hold chunk 0 for all 128 rows; each reads the columns of its own tile.
      mbar_wait(&B.acc_full[1], par1, 0xC02);
      par1 ^= 1u;
      tc_fence_after();
      const int od = P.out_dim;
      if ((kPair ? tsel == 0 : c_first == 0) && q * 32 < od) {
        uint32_t v[32];
        tmem_ld32(lane_taddr + 256u + static_cast<uint32_t>((kPair ? static_cast<int>(crank) * kNR : 0) + w * kWin), v);
        tc_wait_ld();
        const int j = q * 32 + lane;
        if (j < od) {
          const float b3 = __ldg(P.b[3] + j);
#pragma unroll
          for (int r = 0; r < kWin; ++r) {
            const int st = r % C::NS;
            const bool primal = r < C::SPW * C::NS && (st == 0 || (C::kI && st == C::sI));
            outs[(w * kWin + r) * od + j] = __uint_as_float(v[r]) + (primal ? b3 : 0.f);
          }
        }
      }
      tc_fence_before();
      TL_MARK(tl, 0x700u);
      row_warps_sync();
      TL_MARK(tl, 0x710u);
      fwd_loss_stage<C>(P, s0, tile_ok, outs, red, b3sum, t);
      row_warps_sync();   // nobody overwrites the staged outputs (next tile's layer-0 epilogue) while they are read
      TL_MARK(tl, 0x720u);
      if (kPair && tb + tile_stride < n_tiles) {
        // ... nor does the peer, whose layer-0 epilogue of the next tile writes this CTA's rows: tell it
        __syncwarp();
        // relaxed: the loss stage's reads of the staged outputs were consumed before the barrier above, and a release at
        // cluster scope is a GPU-scope membar (~2 K cycles per tile on every row warp)
        if (lane == 0) mbar_arrive_remote_relaxed(xfree_peer);
      }
    }
    // ---- flush the CTA's loss sums and output-bias gradient
    if (t == 0) {
      atomicAdd(&P.losses[1], red[1] * P.inv_B);
      atomicAdd(&P.losses[2], red[2] * P.inv_B);
      atomicAdd(&P.losses[3], red[3] * P.inv_B);
      atomicAdd(&P.losses[0], ((P.kind == DMIP_LOSS_PINN2 ? 0.f : red[1]) + red[2] + red[3]) * P.inv_B);
    }
    if (t < P.out_dim) atomicAdd(&P.grad[P.off_b[3] + t], b3sum[t]);
    TL_CLOSE(tl);
  }
  tcl_teardown(tmem_base, warp);
}

// ------------------------------------------------------------------------------------------------ backward
// Operand of the backward pass's first GEMM: the output adjoints abar (fp32, written by the forward loss stage) of the
// tile's 64 adjoint rows as the MN-major B operand [component j][row] — and the same rows, as they are, as the ADJ_3
// stash block (weight gradient of the output layer).  Padding rows and rows of samples past the batch are zero; the
// matching rows of the IN_0 stash block are zeroed here too (the forward writes only live rows).
template <class C>
__device__ __forceinline__ void bwd_build_input(const TclDev& P, long long tile, bool tile_ok, uint8_t* sIn, int t) {
  // one row x 8 consecutive output components per thread (see fwd_build_input)
  const int row = t & 63, jg = t >> 6;
  const int od = P.out_dim;
  const int w = row >> 5, rw = row & 31;
  const int sj = rw / C::NADJ, a = rw - sj * C::NADJ;
  const long long smp = tile * (2 * C::SPWB) + w * C::SPWB + sj;
  const bool live = tile_ok && sj < C::SPWB && smp < P.B;
  float v[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int j = jg * 8 + e;
    v[e] = (live && j < od) ? P.abar[(smp * C::NADJ + a) * od + j] : 0.f;
  }
  uint32_t hi[4], lo[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) split2(v[2 * e], v[2 * e + 1], hi[e], lo[e]);
  uint8_t* atom = sIn + jg * 1024 + (row & 7) * 2;
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    uint8_t* q = atom + e * 128 + (((row >> 3) ^ e) << 4);
    const uint32_t h2 = hi[e >> 1], l2 = lo[e >> 1];
    *reinterpret_cast<unsigned short*>(q) = static_cast<unsigned short>((e & 1) ? (h2 >> 16) : (h2 & 0xFFFFu));
    *reinterpret_cast<unsigned short*>(q + kInHalf) = static_cast<unsigned short>((e & 1) ? (l2 >> 16) : (l2 & 0xFFFFu));
  }
  if (tile_ok) {
    const size_t o = static_cast<size_t>(tile) * (kTclSmallF * 128) + img_off(static_cast<uint32_t>(row), static_cast<uint32_t>(jg * 8));
    *reinterpret_cast<uint4*>(P.adj_img[3][0] + o) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(P.adj_img[3][1] + o) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    if (!live) {
      *reinterpret_cast<uint4*>(P.in_img[0][0] + o) = make_uint4(0, 0, 0, 0);
      *reinterpret_cast<uint4*>(P.in_img[0][1] + o) = make_uint4(0, 0, 0, 0);
    }
  }
}

// One (layer, chunk, window) item of the backward epilogue: thread = feature k of hidden layer L; the accumulator holds
// hbar (adjoint of the layer's OUTPUT) for the window's adjoint rows.  With phi', phi'' at the stored forward state:
//     zbar_P = phi' hbar_P + phi'' zd_T hbar_T,   zbar_T = phi' hbar_T,   zbar_I = phi'_I hbar_I.
// The derivative state (dmip_tcl.h: st) is fetched with ONE batch of independent loads before the accumulator is
// touched — per-sample dependent loads cost an HBM round trip each (measured: 171 K instead of 60 K cycles per tile).
// Returns this thread's contribution to d loss / d b_L[k] (primal rows only).
template <class C>
__device__ __forceinline__ void bwd_prefetch(const TclDev& P, int L, int k, long long tile, int w, float (&pre)[C::SPWB * C::NADJ]) {
  const float* sst = P.st[L] + k;
  const long long last = P.B - 1;
#pragma unroll
  for (int j = 0; j < C::SPWB; ++j) {
    long long smp = tile * (2 * C::SPWB) + w * C::SPWB + j;
    smp = smp < last ? smp : last;                   // rows past the batch read a valid sample and are masked later
#pragma unroll
    for (int a = 0; a < C::NADJ; ++a) pre[j * C::NADJ + a] = __ldg(sst + (smp * C::NADJ + a) * 512);
  }
}

// accumulator (hbar) -> zbar rows in v[]; returns the bias-gradient contribution
template <class C>
__device__ __forceinline__ float bwd_math(const TclDev& P, uint32_t taddr, long long tile, bool tile_ok, int w,
                                          const float (&pre)[C::SPWB * C::NADJ], uint32_t (&v)[32]) {
  tmem_ld32(taddr, v);
  tc_wait_ld();
  float bs = 0.f;
#pragma unroll
  for (int j = 0; j < C::SPWB; ++j) {
    const int base = j * C::NADJ;
    const long long smp = tile * (2 * C::SPWB) + w * C::SPWB + j;
    const bool live = tile_ok && smp < P.B;
    const float p1 = pre[base];
    float zP = p1 * __uint_as_float(v[base]), zI = 0.f, zT = 0.f;
    if (C::kT) {
      const float hbT = __uint_as_float(v[base + 1 + C::kI]);
      zP = fmaf(pre[base + 1 + C::kI], hbT, zP);
      zT = p1 * hbT;
    }
    if (C::kI) zI = pre[base + 1] * __uint_as_float(v[base + 1]);
    if (!live) zP = zI = zT = 0.f;
    bs += zP + zI;
    v[base] = __float_as_uint(zP);
    if (C::kI) v[base + 1] = __float_as_uint(zI);
    if (C::kT) v[base + 1 + C::kI] = __float_as_uint(zT);
  }
#pragma unroll
  for (int r = C::SPWB * C::NADJ; r < kWin; ++r) v[r] = 0u;
  return bs;
}

// zbar rows -> ADJ_L stash block (all 32 rows of the window, zeros included; the padding rows of IN_{L+1} are zeroed as
// well) and, for L > 0, the B operand of the next GEMM
template <class C>
__device__ __forceinline__ void bwd_store(const TclDev& P, int L, bool to_smem, int k, long long tile, bool tile_ok, int w,
                                          const uint32_t (&v)[32], uint32_t hdst, uint32_t rmbar, uint64_t* hready,
                                          uint32_t hready_leader, int lane) {
  const uint32_t kterm = (static_cast<uint32_t>(k) >> 6) * 8192u + (static_cast<uint32_t>(k) & 7u) * 2u;
  const uint32_t kchunk = (static_cast<uint32_t>(k) & 63u) >> 3;
  const size_t blk = static_cast<size_t>(tile) * (512 * 128) + kterm;
  auto row_off = [&](uint32_t r) { return (r >> 3) * 1024u + (r & 7u) * 128u + ((kchunk ^ (r & 7u)) << 4); };
  if (to_smem) {
    const uint32_t hrow = hdst + (static_cast<uint32_t>(k) >> 3) * 1024u + (static_cast<uint32_t>(k) & 7u) * 128u;
    const uint32_t line = static_cast<uint32_t>(k) & 7u;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      uint32_t hi[4], lo[4];
#pragma unroll
      for (int e = 0; e < 4; ++e)
        split2(__uint_as_float(v[i * 8 + 2 * e]), __uint_as_float(v[i * 8 + 2 * e + 1]), hi[e], lo[e]);
      const uint32_t co = ((static_cast<uint32_t>(w * 4 + i) ^ line) << 4);
      st_operand_v4(hrow + co, hi[0], hi[1], hi[2], hi[3], rmbar);
      st_operand_v4(hrow + kHHalf + co, lo[0], lo[1], lo[2], lo[3], rmbar);
    }
    // the next GEMM may read these K-blocks now; the global stash stores below are off its critical path
    if (rmbar == 0u) {   // remote rows (st.async): the peer's receiver warp tells the issuer
      fence_operand_stores();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) arrive_issuer(hready, hready_leader);
    }
  }
  if (tile_ok) {
    const uint32_t wo = static_cast<uint32_t>(w) * 4096u;           // window w starts 4 row-groups (4 KB) into the block
    uint8_t* ahi = P.adj_img[L][0] + blk + wo;
    uint8_t* alo = P.adj_img[L][1] + blk + wo;
    uint8_t* ihi = P.in_img[L + 1][0] + blk + wo;
    uint8_t* ilo = P.in_img[L + 1][1] + blk + wo;
    const uint32_t kc4 = kchunk << 4;                               // swizzle term: one XOR with an immediate per row
    const long long s_first = tile * (2 * C::SPWB) + w * C::SPWB;
    const bool full = s_first + C::SPWB <= P.B;                     // warp-uniform: no row of a live sample is missing
    // rows in the order (r & 7) outer, (r >> 3) inner: one swizzled chunk offset is live at a time
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const uint32_t xo = i * 128u + (kc4 ^ (static_cast<uint32_t>(i) << 4));
#pragma unroll
      for (int q = 0; q < kWin / 8; ++q) {
        const int r = q * 8 + i;
        unsigned short hi, lo;
        split1(__uint_as_float(v[r]), hi, lo);
        const uint32_t o = q * 1024u + xo;
        *reinterpret_cast<unsigned short*>(ahi + o) = hi;
        *reinterpret_cast<unsigned short*>(alo + o) = lo;
        const int j = r / C::NADJ;
        const bool dead = j >= C::SPWB || (!full && s_first + j >= P.B);
        if (dead) {
          *reinterpret_cast<unsigned short*>(ihi + o) = 0;
          *reinterpret_cast<unsigned short*>(ilo + o) = 0;
        }
      }
    }
  }
}

// kGradIn: a fourth GEMM, xbar = zbar_0 W0 (A = W0^T, one 128-row chunk of input columns), gives the gradient w.r.t. the
// net's inputs (dmip_mlp_backward and, from the P rows, dmip_mlp_double_backward; the losses do not need it: grad_x of the
// Score-FPE term is a constant, SURVEY.md Q9).
template <class C, bool kGradIn>
__global__ void __launch_bounds__(kThreads, 1) k_tcl_bwd(const __grid_constant__ TclDev P) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const Bars B = make_bars(smem);
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const uint32_t tmem_base = tcl_setup(smem, B, warp, lane);
  const uint32_t crank = kCluster > 1 ? cluster_ctarank() : 0u;
  const uint16_t cmask = static_cast<uint16_t>((1u << kCluster) - 1u);
  const int n_tiles = keep(static_cast<int>(P.n_tiles_bwd));
  const int tile_first = static_cast<int>(blockIdx.x / kCluster) * kCluster;
  const int tile_stride = keep(static_cast<int>(gridDim.x));

  if (warp >= kNumRowWarps) {
    reg_dealloc<kRegsSmall>();
    if (kGradIn)
      tcl_service_warps<4, 1>(warp, keep(P.stages_bwd), kTclBwdStagesIn, keep(P.k0steps_bwd), tile_first, n_tiles, tile_stride,
                              smem, tmem_base, B, crank, cmask);
    else
      tcl_service_warps<3, 4>(warp, keep(P.stages_bwd), kTclBwdStages, keep(P.k0steps_bwd), tile_first, n_tiles, tile_stride,
                              smem, tmem_base, B, crank, cmask);
  } else {
    reg_alloc<kRegsRow>();
    const int q = warp & 3, cgp = warp >> 2;
    const int w = cgp & 1;                                             // window; chunks / tile as in k_tcl_fwd
    const int c_first = kPair ? static_cast<int>(crank) : cgp >> 1;
    const int tsel = kPair ? cgp >> 1 : static_cast<int>(crank);
    const int t = threadIdx.x;
    const uint32_t lane_taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const uint32_t hdst = (kPair && tsel != static_cast<int>(crank)) ? mapa_u32(smem + kOffHhi, static_cast<uint32_t>(tsel))
                                                                      : smem_u32(smem + kOffHhi);
    const uint32_t in_ready_leader = kPair ? mapa_u32(B.in_ready, 0) : 0u;
    const uint32_t hready_leader = kPair ? mapa_u32(&B.hready[0], 0) : 0u;
    const uint32_t rready_dst = (kPair && tsel != static_cast<int>(crank)) ? mapa_u32(&B.rready[0], static_cast<uint32_t>(tsel)) : 0u;
    uint32_t par = 0;   // bit s: phase of acc_full[s]
    uint32_t gc = 0;    // running GEMM counter (three GEMMs per tile: the TMEM half of a GEMM is gc & 1, as in tcl_issuer)
    float bsum[3][2] = {{0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}};   // bias gradients of layers 2, 1, 0 for this thread's two features
    {
      const bool ok = tile_first + static_cast<int>(crank) < n_tiles;
      bwd_build_input<C>(P, tile_first + static_cast<int>(crank), ok, smem + kOffIn, t);
      fence_operand_stores();
      __syncwarp();
      if (lane == 0) arrive_issuer(B.in_ready, in_ready_leader);
    }
    for (int tb = tile_first; tb < n_tiles; tb += tile_stride) {
      const bool tile_ok = tb + static_cast<int>(crank) < n_tiles;     // this CTA's own tile
      const long long tile = tb + static_cast<int>(crank);
      const long long etile = tb + tsel;                               // the tile whose rows this warp's items hold
      const bool etile_ok = etile < n_tiles;
      // accumulator columns of this warp's two items inside a TMEM half
      const uint32_t col0 = kPair ? static_cast<uint32_t>(tsel * kNR + w * kWin) : static_cast<uint32_t>(c_first * kNR + w * kWin);
      constexpr uint32_t kColStep = 2 * kNR;                           // second item: chunk c_first + 2
#pragma unroll
      for (int g = 0; g < 3; ++g) {
        const int L = 2 - g;
        const uint32_t set = gc & 1u;
        ++gc;
        const int k0 = c_first * 128 + q * 32 + lane, k1 = k0 + 256;     // this thread's two features (chunks c_first, c_first + 2)
        // software pipeline: the derivative state of an item is in flight while the GEMM finishes / while the previous
        // item's results are stored
        float pre[C::SPWB * C::NADJ];
        uint32_t v[32];
        bwd_prefetch<C>(P, L, k0, etile, w, pre);
        mbar_wait(&B.acc_full[set], (par >> set) & 1u, 0xD00 + set);
        par ^= 1u << set;
        tc_fence_after();
        const uint32_t t0 = lane_taddr + set * 256u + col0;
        bsum[g][0] += bwd_math<C>(P, t0, etile, etile_ok, w, pre, v);
        bwd_prefetch<C>(P, L, k1, etile, w, pre);
        bwd_store<C>(P, L, L != 0 || kGradIn, k0, etile, etile_ok, w, v, hdst, rready_dst ? rready_dst + c_first * 8u : 0u, &B.hready[c_first],
                     hready_leader + static_cast<uint32_t>(c_first) * 8u, lane);
        bsum[g][1] += bwd_math<C>(P, t0 + kColStep, etile, etile_ok, w, pre, v);
        bwd_store<C>(P, L, L != 0 || kGradIn, k1, etile, etile_ok, w, v, hdst, rready_dst ? rready_dst + (c_first + 2) * 8u : 0u, &B.hready[c_first + 2],
                     hready_leader + static_cast<uint32_t>(c_first + 2) * 8u, lane);
        if (g == 1 && tb + tile_stride < n_tiles) {
          const int nt = tb + tile_stride + static_cast<int>(crank);
          bwd_build_input<C>(P, nt, nt < n_tiles, smem + kOffIn, t);
          fence_operand_stores();
          __syncwarp();
          if (lane == 0) arrive_issuer(B.in_ready, in_ready_leader);
        }
      }
      if (kGradIn) {
        // ---- gradient w.r.t. the inputs: accumulator chunk 0 = (input column, row); rows are (sample, adjoint stream)
        // pairs, and the P rows hold the result (double backward: the T rows' input adjoint would be d / dv, not needed).
        // Pair mode: both CTAs hold the chunk for all 128 rows; each reads the columns of its own tile.
        const uint32_t set = gc & 1u;
        ++gc;
        mbar_wait(&B.acc_full[set], (par >> set) & 1u, 0xD10 + set);
        par ^= 1u << set;
        tc_fence_after();
        if ((kPair ? tsel == 0 : c_first == 0) && q * 32 < P.in_dim) {
          uint32_t v[32];
          tmem_ld32(lane_taddr + set * 256u + static_cast<uint32_t>((kPair ? static_cast<int>(crank) * kNR : 0) + w * kWin), v);
          tc_wait_ld();
          const int k = q * 32 + lane;
          if (k < P.in_dim && tile_ok) {
#pragma unroll
            for (int r = 0; r < C::SPWB * C::NADJ; r += C::NADJ) {
              const long long smp = tile * (2 * C::SPWB) + w * C::SPWB + r / C::NADJ;
              if (smp < P.B) P.grad_in[smp * P.in_dim + k] = __uint_as_float(v[r]);
            }
          }
        }
        tc_fence_before();
        // the next tile's first epilogue overwrites the activation region this GEMM read: it has retired (acc_full)
      }
    }
#pragma unroll
    for (int g = 0; g < 3; ++g)
#pragma unroll
      for (int ci = 0; ci < 2; ++ci) {
        const int k = (c_first + 2 * ci) * 128 + q * 32 + lane;
        red_add_f32(&P.grad[P.off_b[2 - g] + k], bsum[g][ci]);
      }
    tc_fence_before();
  }
  tcl_teardown(tmem_base, warp);
}

// ------------------------------------------------------------------------------------------------ weight gradients
// dW[m][n] += sum_r A[r][m] B[r][n] over the 64-row stash blocks [blk0, blk1): A and B are MN-major bf16 hi/lo images
// (dmip_tcl.h), bulk-copied as they are; per block 4 K = 16 steps x 3 split products of one M = 128, N = kN instruction;
// the fp32 accumulator (kN TMEM columns) lives for the CTA's whole row range and is added to the flat gradient with
// fp32 atomics at the end (split-K across CTAs).  grid = (M chunks x N chunks, splits).
struct WgradJob {
  const uint8_t *a_hi, *a_lo, *b_hi, *b_lo;
  int FA, FB;            // features of the A / B images
  int n_mchunks, n_nchunks, n_cols;   // N of one instruction = n_cols (64 or 256), B chunk cn = features [cn n_cols, +n_cols)
  long long n_blocks, blocks_per_split;
  float* dW;             // destination; element (m, n) of the product goes to dW[m * ldw + n], or dW[n * ldw + m] if transposed
  int ldw, transposed;
  int m_valid, n_valid;  // rows / columns of the product that exist in dW
};

constexpr int kWgThreads = 192;      // warps 0-3 epilogue, 4 producer, 5 MMA issuer
constexpr int kWgStageA = 32768;     // A hi + A lo: 2 x (128 features x 64 rows x bf16)

template <int kN>
__global__ void __launch_bounds__(kWgThreads, 1) k_tcl_wgrad(const __grid_constant__ WgradJob J) {
  constexpr int kStageB = 2 * kN * 128;                  // B hi + B lo
  constexpr int kStageBytes = kWgStageA + kStageB;
  constexpr int kNS = kN == 256 ? 2 : 4;                 // ring depth
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kNS * kStageBytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + kNS;
  uint64_t* done = bars + 2 * kNS;
  uint32_t* holder = reinterpret_cast<uint32_t*>(bars + 2 * kNS + 1);
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  if ((smem_u32(smem) & 1023u) != 0u) __trap();
  if (threadIdx.x == 0) {
    for (int i = 0; i < kNS; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(done, 1);
    fence_barrier_init();
  }
  if (warp == 5) tmem_alloc<kN>(holder);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *holder, 0);
  const int cm = blockIdx.x / J.n_nchunks, cn = blockIdx.x % J.n_nchunks;
  const long long blk0 = static_cast<long long>(blockIdx.y) * J.blocks_per_split;
  const long long blk1 = min(J.n_blocks, blk0 + J.blocks_per_split);

  if (warp == 4) {
    int s = 0;
    uint32_t ph = 0;
    const size_t strideA = static_cast<size_t>(J.FA) * 128, strideB = static_cast<size_t>(J.FB) * 128;
    const uint8_t* a_hi = J.a_hi + static_cast<size_t>(cm) * 16384;
    const uint8_t* a_lo = J.a_lo + static_cast<size_t>(cm) * 16384;
    const uint8_t* b_hi = J.b_hi + static_cast<size_t>(cn) * (kN * 128);
    const uint8_t* b_lo = J.b_lo + static_cast<size_t>(cn) * (kN * 128);
    for (long long b = blk0; b < blk1; ++b) {
      mbar_wait(&empty[s], ph ^ 1u, 0xE00 + s);
      if (elect_one()) {
        uint8_t* st = smem + s * kStageBytes;
        mbar_arrive_expect_tx(&full[s], kStageBytes);
        bulk_g2s(st, a_hi + b * strideA, 16384, &full[s]);
        bulk_g2s(st + 16384, a_lo + b * strideA, 16384, &full[s]);
        bulk_g2s(st + kWgStageA, b_hi + b * strideB, kN * 128, &full[s]);
        bulk_g2s(st + kWgStageA + kN * 128, b_lo + b * strideB, kN * 128, &full[s]);
      }
      __syncwarp();
      if (++s == kNS) { s = 0; ph ^= 1u; }
    }
  } else if (warp == 5) {
    int s = 0;
    uint32_t ph = 0;
    const uint32_t base16 = (smem_u32(smem) & 0x3FFFFu) >> 4;
    // both operands MN-major: 64-feature groups 8 KB apart, 8-row (K) groups 1 KB apart
    const uint64_t desc = umma_smem_desc(0, 8192, 1024);   // address field 0: OR-ed in per instruction (LBO sits in the LOW word)
    constexpr uint32_t idesc = umma_idesc_bf16_major(128, kN, 1, 1);
    for (long long b = blk0; b < blk1; ++b) {
      mbar_wait(&full[s], ph, 0xE10 + s);
      tc_fence_after();
      const uint32_t a16 = base16 + static_cast<uint32_t>(s) * (kStageBytes >> 4);
      const uint32_t b16 = a16 + (kWgStageA >> 4);
      if (elect_one()) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {   // K = 16 rows = two 8-row groups = 2 KB
          umma_ss(tmem_base, desc | (a16 + j * 128), desc | (b16 + j * 128), idesc, (b > blk0 || j > 0) ? 1u : 0u);
          umma_ss(tmem_base, desc | (a16 + j * 128), desc | (b16 + ((kN * 128) >> 4) + j * 128), idesc, 1u);
          umma_ss(tmem_base, desc | (a16 + 1024 + j * 128), desc | (b16 + j * 128), idesc, 1u);
        }
        tc_commit(&empty[s]);
        if (b == blk1 - 1) tc_commit(done);
      }
      __syncwarp();
      if (++s == kNS) { s = 0; ph ^= 1u; }
    }
  } else if (blk1 > blk0) {
    // epilogue warps 0-3: lane = row m of the product
    mbar_wait(done, 0, 0xE20);
    tc_fence_after();
    const int m = cm * 128 + warp * 32 + lane;
    const uint32_t lane_taddr = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
#pragma unroll 1
    for (int c0 = 0; c0 < kN; c0 += 32) {
      uint32_t v[32];
      tmem_ld32(lane_taddr + c0, v);
      tc_wait_ld();
      if (m < J.m_valid) {
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          const int n = cn * kN + c0 + e;
          if (n < J.n_valid) {
            float* dst = J.transposed ? J.dW + static_cast<size_t>(n) * J.ldw + m : J.dW + static_cast<size_t>(m) * J.ldw + n;
            red_add_f32(dst, __uint_as_float(v[e]));
          }
        }
      }
    }
    tc_fence_before();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) {
    tc_fence_after();
    tmem_dealloc<kN>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------ weight images
// One 16 KB stage per block: 128 features x 64 k of W (forward) or W^T (backward), hi or lo part, K-major, 128B swizzle.
__global__ void __launch_bounds__(256) k_tcl_pack(const __grid_constant__ TclDev P) {
  int st = blockIdx.x;
  const bool bwd = st >= kTclFwdStages;
  if (bwd) st -= kTclFwdStages;
  uint8_t* dst = const_cast<uint8_t*>(bwd ? P.stages_bwd : P.stages_fwd) + static_cast<size_t>(st) * kStage;
  int g, c, kb, part;
  if (st < 8) { g = 0; c = st >> 1; kb = 0; part = st & 1; }
  else if (st < 72) { g = 1; const int i = st - 8; kb = i >> 3; c = (i >> 1) & 3; part = i & 1; }
  else if (st < 136) { g = 2; const int i = st - 72; kb = i >> 3; c = (i >> 1) & 3; part = i & 1; }
  else { g = 3; const int i = st - 136; kb = i >> 1; c = 0; part = i & 1; }   // forward: W3; backward: W0^T (input gradient)
  for (int e = threadIdx.x; e < 128 * 64; e += 256) {
    const int r = e >> 6, kk = e & 63;
    const int m = c * 128 + r, k = kb * 64 + kk;
    float v = 0.f;
    if (!bwd) {
      // forward: A = W_g, M = output feature m, K = input feature k
      if (g == 0) { if (k < P.in_dim) v = P.W[0][static_cast<size_t>(m) * P.in_dim + k]; }
      else if (g == 3) { if (m < P.out_dim) v = P.W[3][static_cast<size_t>(m) * 512 + k]; }
      else v = P.W[g][static_cast<size_t>(m) * 512 + k];
    } else {
      // backward: A = W^T: M = input feature m of the layer, K = its output feature k (GEMM 0: W3^T, 1: W2^T, 2: W1^T)
      if (g == 0) { if (k < P.out_dim) v = P.W[3][static_cast<size_t>(k) * 512 + m]; }
      else if (g == 3) { if (m < P.in_dim) v = P.W[0][static_cast<size_t>(k) * P.in_dim + m]; }   // W0^T: M = input column
      else v = P.W[3 - g][static_cast<size_t>(k) * 512 + m];
    }
    unsigned short hi, lo;
    split1(v, hi, lo);
    *reinterpret_cast<unsigned short*>(dst + sw128_offset(static_cast<uint32_t>(r), static_cast<uint32_t>(kk), kStage)) = part ? lo : hi;
  }
}

int g_tcl_sm = 0;
bool g_tcl_ready[64] = {};

template <class C>
int set_attr() {
  DMIP_CHECK_CUDA(cudaFuncSetAttribute(k_tcl_fwd<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
  DMIP_CHECK_CUDA(cudaFuncSetAttribute((k_tcl_bwd<C, false>), cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
  return DMIP_OK;
}

constexpr int wg_smem(int n) { return (n == 256 ? 2 : 4) * (kWgStageA + 2 * n * 128) + 128 + 1024; }

// the compiled stream configurations: DSM / DPS likelihood | cScoreFPE, adjoint-route PDE | the same with the initial
// condition | DSM_PDE and PINN with exact Score-FPE (d = 2, 3, 4) | DPS prior (Jacobian, d = 3)
#define DMIP_TCL_CONFIGS(X) \
  X(0, 0, 0, 0) X(0, 1, 0, 0) X(1, 1, 0, 0) X(0, 1, 2, 1) X(1, 1, 2, 1) X(1, 1, 3, 1) X(1, 1, 4, 1) X(0, 0, 3, 0)

int tcl_init() {
  int dev = 0;
  DMIP_CHECK_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || !g_tcl_ready[dev]) {
    DMIP_CHECK_CUDA(cudaDeviceGetAttribute(&g_tcl_sm, cudaDevAttrMultiProcessorCount, dev));
    int rc;
#define X(i, t, n, q) if ((rc = set_attr<Cfg<i, t, n, q>>())) return rc;
    DMIP_TCL_CONFIGS(X)
#undef X
    DMIP_CHECK_CUDA(cudaFuncSetAttribute((k_tcl_bwd<Cfg<0, 0, 0, 0>, true>), cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    DMIP_CHECK_CUDA(cudaFuncSetAttribute((k_tcl_bwd<Cfg<0, 1, 0, 0>, true>), cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    DMIP_CHECK_CUDA(cudaFuncSetAttribute(k_tcl_wgrad<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, wg_smem(256)));
    DMIP_CHECK_CUDA(cudaFuncSetAttribute(k_tcl_wgrad<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, wg_smem(64)));
    if (dev >= 0 && dev < 64) g_tcl_ready[dev] = true;
  }
  return DMIP_OK;
}

template <class K>
int launch_clustered(K kernel, long long n_tiles, const TclDev& P, cudaStream_t s) {
  if (n_tiles <= 0) return DMIP_OK;
  DMIP_REQUIRE(n_tiles < (1LL << 31), "too many tiles in one call (%lld)", n_tiles);
  const long long want = (n_tiles + kCluster - 1) / kCluster, have = g_tcl_sm / kCluster;
  const long long n_clusters = want < have ? want : have;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(n_clusters * kCluster));
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = kSmemBytes;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kCluster;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  DMIP_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kernel, P));
  DMIP_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return DMIP_OK;
}

}  // namespace

void tcl_debug_set_timeline(unsigned long long* buf, int cap) {
#ifdef DMIP_JOBMARKS
  cudaMemcpyToSymbol(g_tcl_tl, &buf, sizeof(buf));
  cudaMemcpyToSymbol(g_tcl_tl_cap, &cap, sizeof(cap));
#else
  (void)buf;
  (void)cap;
#endif
}

bool tcl_streams_supported(const TclStreams& s) {
#define X(i, t, n, q) if (s.has_I == i && s.has_T == t && s.n_tan == n && s.has_Q == q) return true;
  DMIP_TCL_CONFIGS(X)
#undef X
  return false;
}

size_t tcl_image_bytes() { return static_cast<size_t>(kTclFwdStages + kTclBwdStagesIn) * kStage; }

int tcl_launch_pack(const TclDev& P, cudaStream_t s) {
  k_tcl_pack<<<kTclFwdStages + kTclBwdStagesIn, 256, 0, s>>>(P);
  DMIP_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return DMIP_OK;
}

int tcl_launch_fwd(const TclDev& P, cudaStream_t s) {
  int rc = tcl_init();
  if (rc) return rc;
#define X(i, t, n, q) \
  if (P.has_I == i && P.has_T == t && P.n_tan == n && P.has_Q == q) return launch_clustered(k_tcl_fwd<Cfg<i, t, n, q>>, P.n_tiles_fwd, P, s);
  DMIP_TCL_CONFIGS(X)
#undef X
  set_error("tcgen05 loss path: stream configuration not compiled in");
  return DMIP_EINVAL;
}

int tcl_launch_bwd(const TclDev& P, cudaStream_t s) {
  int rc = tcl_init();
  if (rc) return rc;
  if (P.grad_in != nullptr) {
    DMIP_REQUIRE(P.has_I == 0 && P.n_tan == 0 && P.has_Q == 0,
                 "input gradients are computed for the plain net pass and its double backward only");
    if (P.has_T) return launch_clustered(k_tcl_bwd<Cfg<0, 1, 0, 0>, true>, P.n_tiles_bwd, P, s);
    return launch_clustered(k_tcl_bwd<Cfg<0, 0, 0, 0>, true>, P.n_tiles_bwd, P, s);
  }
#define X(i, t, n, q) \
  if (P.has_I == i && P.has_T == t && P.n_tan == n && P.has_Q == q) \
    return launch_clustered(k_tcl_bwd<Cfg<i, t, n, q>, false>, P.n_tiles_bwd, P, s);
  DMIP_TCL_CONFIGS(X)
#undef X
  set_error("tcgen05 loss path: stream configuration not compiled in");
  return DMIP_EINVAL;
}

int tcl_launch_wgrad(const TclDev& P, cudaStream_t s) {
  int rc = tcl_init();
  if (rc) return rc;
  const long long n_blocks = P.n_tiles_bwd;
  if (n_blocks <= 0) return DMIP_OK;
  long long off = 0;   // float offset of W_l in the flat gradient
  int k = P.in_dim;
  for (int l = 0; l < 4; ++l) {
    const int n = l == 3 ? P.out_dim : 512;
    WgradJob J = {};
    J.n_blocks = n_blocks;
    J.dW = P.grad + off;
    J.ldw = k;
    if (l == 3) {
      // few outputs: the wide side (inputs of the layer) is the M side, the product is stored transposed
      J.a_hi = P.in_img[3][0]; J.a_lo = P.in_img[3][1]; J.FA = 512;
      J.b_hi = P.adj_img[3][0]; J.b_lo = P.adj_img[3][1]; J.FB = kTclSmallF;
      J.n_mchunks = 4; J.n_nchunks = 1; J.n_cols = 64;
      J.transposed = 1; J.m_valid = 512; J.n_valid = n;
    } else {
      J.a_hi = P.adj_img[l][0]; J.a_lo = P.adj_img[l][1]; J.FA = 512;
      J.b_hi = P.in_img[l][0]; J.b_lo = P.in_img[l][1]; J.FB = l == 0 ? kTclSmallF : 512;
      J.n_mchunks = 4; J.n_nchunks = l == 0 ? 1 : 2; J.n_cols = l == 0 ? 64 : 256;
      J.transposed = 0; J.m_valid = 512; J.n_valid = k;
    }
    const int tiles = J.n_mchunks * J.n_nchunks;
    long long splits = g_tcl_sm / tiles;
    if (splits > n_blocks) splits = n_blocks;
    if (splits < 1) splits = 1;
    J.blocks_per_split = (n_blocks + splits - 1) / splits;
    splits = (n_blocks + J.blocks_per_split - 1) / J.blocks_per_split;
    dim3 grid(static_cast<unsigned>(tiles), static_cast<unsigned>(splits));
    if (J.n_cols == 256) k_tcl_wgrad<256><<<grid, kWgThreads, wg_smem(256), s>>>(J);
    else k_tcl_wgrad<64><<<grid, kWgThreads, wg_smem(64), s>>>(J);
    DMIP_CHECK_CUDA(cudaGetLastError());
    count_launch();
    off += static_cast<long long>(n) * k + n;
    k = n;
  }
  return DMIP_OK;
}

}  // namespace dmip
