// dmip_tile.cuh — the fp32 32-row tile engine shared by the FFMA kernels (fp32 sampler / forward, losses, surrogate,
// Metropolis): activations live in shared memory transposed ([k][row], row stride kLd), a layer is a 32 x N x K
// register-tiled FFMA GEMM against weights stored [contraction][output] in global memory (L2/L1 resident).  The host
// side prepares a net for it with tile_net_check / tile_net_bytes / tile_net_stage (end of this file).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "dmip_common.h"

namespace dmip {
namespace {

constexpr int kRows = 32;
constexpr int kLd = 36;
constexpr int kMaxW = 512;
constexpr int kThreadsL = 512;   // 16 warps: 4 per scheduler hide the L1/L2 latency of the weight loads

// out[n*kLd + r] = sum_k in[k*kLd + r] * Wt[k*N + n], r < 32, n < N.  512 threads: thread (rg, ng) owns rows 8 rg .. 8 rg + 7
// and columns ng + 128 i, i < 4; the operands of step k+1 are fetched while step k's 32 FMAs issue.  Ends with
// __syncthreads().
__device__ void tile_gemm_direct(const float* in, float* out, const float* __restrict__ Wt, int K, int N) {
  const int t = threadIdx.x;
  const int rg = t >> 7, ng = t & 127;
  for (int nb = 0; nb < N; nb += 512) {
    float acc[8][4];
#pragma unroll
    for (int r = 0; r < 8; ++r)
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[r][i] = 0.f;
    const int ncols = (N - nb - ng + 127) >> 7;   // columns of this thread inside [nb, nb + 512)
    if (ncols > 0) {
      const float* wp = Wt + nb + ng;
      float4 a0 = *reinterpret_cast<const float4*>(in + rg * 8);
      float4 a1 = *reinterpret_cast<const float4*>(in + rg * 8 + 4);
      float w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) w[i] = (i < ncols) ? __ldg(wp + 128 * i) : 0.f;
      for (int k = 0; k < K; ++k) {
        const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        float wc[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) wc[i] = w[i];
        if (k + 1 < K) {   // prefetch step k+1
          a0 = *reinterpret_cast<const float4*>(in + (k + 1) * kLd + rg * 8);
          a1 = *reinterpret_cast<const float4*>(in + (k + 1) * kLd + rg * 8 + 4);
          const float* wn = wp + static_cast<size_t>(k + 1) * N;
#pragma unroll
          for (int i = 0; i < 4; ++i) w[i] = (i < ncols) ? __ldg(wn + 128 * i) : 0.f;
        }
#pragma unroll
        for (int r = 0; r < 8; ++r)
#pragma unroll
          for (int i = 0; i < 4; ++i) acc[r][i] = fmaf(a[r], wc[i], acc[r][i]);
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int n = nb + ng + 128 * i;
      if (n < N) {
#pragma unroll
        for (int r = 0; r < 8; ++r) out[n * kLd + rg * 8 + r] = acc[r][i];
      }
    }
  }
  __syncthreads();
}


// ---- staged variant: the weights stream through shared memory in 16-k slabs (cp.async, double buffered), so their L2
// latency is paid one slab (16 k-steps) ahead instead of one k-step ahead, and every thread reads its four weights with
// one conflict-free LDS.128.  Thread (rg, ng) owns R rows and columns 4 ng .. 4 ng + 3; N = 64 R (512 or 256).  A warp
// covers ALL 32 rows x 4 R columns (lane = row group x column group), so per k-step it touches 128 B of activations
// and 16 R B of weights: 3 shared-memory wavefronts per 32 FFMA instead of 6 with one row group per warp.
constexpr int kSlabK = 16;
constexpr int kSlabPad = 8;                                   // slab row stride N + 8: conflict-free fragment loads
constexpr int kWbufFloats = 2 * kSlabK * (kMaxW + kSlabPad);  // 65 KB

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst))),
               "l"(gsrc)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int kN>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(kN) : "memory"); }

template <int R>
__device__ void tile_gemm_staged(const float* in, float* out, const float* __restrict__ Wt, int K, float* wbuf) {
  constexpr int N = 64 * R;              // 512 threads x (4 columns x R rows) = 32 rows x N columns
  constexpr int kGroups = N / 4;         // column groups
  const int t = threadIdx.x;
  const int rg = (t & 31) / R, ng = (t >> 5) * R + (t & 31) % R;   // 32 / R row groups x R column groups per warp
  static_assert(kGroups == (kThreadsL / 32) * R, "16 warps x R column groups cover the N / 4 groups");
  float acc[R][4];
#pragma unroll
  for (int r = 0; r < R; ++r)
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[r][i] = 0.f;
  const int n_slabs = K / kSlabK;
  constexpr int kChunks = kSlabK * N / 4;   // 16-byte chunks per slab
  auto issue = [&](int s) {
    const float* src = Wt + static_cast<size_t>(s) * kSlabK * N;
    float* dst = wbuf + (s & 1) * kSlabK * N;
    for (int c = t; c < kChunks; c += kThreadsL) cp_async16(dst + c * 4, src + c * 4);
    cp_async_commit();
  };
  issue(0);
  for (int s = 0; s < n_slabs; ++s) {
    if (s + 1 < n_slabs) {
      issue(s + 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();   // slab s has landed for every thread
    const float* w = wbuf + (s & 1) * kSlabK * N + ng * 4;
    const float* a = in + s * kSlabK * kLd + rg * R;
#pragma unroll
    for (int k = 0; k < kSlabK; ++k) {
      const float4 wv = *reinterpret_cast<const float4*>(w + k * N);
      float av[R];
      if (R == 8) {
        const float4 a0 = *reinterpret_cast<const float4*>(a + k * kLd);
        const float4 a1 = *reinterpret_cast<const float4*>(a + k * kLd + 4);
        av[0] = a0.x; av[1] = a0.y; av[2] = a0.z; av[3] = a0.w;
        av[R > 4 ? 4 : 0] = a1.x; av[R > 4 ? 5 : 0] = a1.y; av[R > 4 ? 6 : 0] = a1.z; av[R > 4 ? 7 : 0] = a1.w;
      } else {
        const float4 a0 = *reinterpret_cast<const float4*>(a + k * kLd);
        av[0] = a0.x; av[1] = a0.y; av[2] = a0.z; av[3] = a0.w;
      }
#pragma unroll
      for (int r = 0; r < R; ++r) {
        acc[r][0] = fmaf(av[r], wv.x, acc[r][0]);
        acc[r][1] = fmaf(av[r], wv.y, acc[r][1]);
        acc[r][2] = fmaf(av[r], wv.z, acc[r][2]);
        acc[r][3] = fmaf(av[r], wv.w, acc[r][3]);
      }
    }
    __syncthreads();   // everyone is done with this buffer before slab s+2 is copied into it
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float* o = out + (ng * 4 + i) * kLd + rg * R;
    if (R == 8) {
      *reinterpret_cast<float4*>(o) = make_float4(acc[0][i], acc[1][i], acc[2][i], acc[3][i]);
      *reinterpret_cast<float4*>(o + 4) = make_float4(acc[R > 4 ? 4 : 0][i], acc[R > 4 ? 5 : 0][i], acc[R > 4 ? 6 : 0][i], acc[R > 4 ? 7 : 0][i]);
    } else {
      *reinterpret_cast<float4*>(o) = make_float4(acc[0][i], acc[1][i], acc[2][i], acc[3][i]);
    }
  }
  __syncthreads();
}

// ---- skinny outputs (N <= 32 with a long contraction: the nets' last layer, the first layer of a reverse sweep).  The
// direct path would leave all but 4 N threads idle and walk K serially behind one global load per step (ncu: 30 % of
// k_jets_fwd's warp samples sat at its closing barrier).  Here a row's contraction is cut into 16 k-slices held by one
// half-warp and summed with shuffles; the weights (<= 64 KB) are L1 hits.
__device__ void tile_gemm_skinny(const float* in, float* out, const float* __restrict__ Wt, int K, int N) {
  const int t = threadIdx.x;
  const int r = t >> 4, ks = t & 15;   // 32 rows x 16 k-slices
  for (int nb = 0; nb < N; nb += 8) {
    const int nn = N - nb < 8 ? N - nb : 8;
    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.f;
    for (int k = ks; k < K; k += 16) {
      const float a = in[k * kLd + r];
      const float* w = Wt + static_cast<size_t>(k) * N + nb;
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (i < nn) acc[i] = fmaf(a, __ldg(w + i), acc[i]);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float v = acc[i];
      v += __shfl_xor_sync(0xffffffffu, v, 8);
      v += __shfl_xor_sync(0xffffffffu, v, 4);
      v += __shfl_xor_sync(0xffffffffu, v, 2);
      v += __shfl_xor_sync(0xffffffffu, v, 1);
      if (ks == 0 && i < nn) out[(nb + i) * kLd + r] = v;
    }
  }
  __syncthreads();
}

// ---- tensor-core variant of the staged GEMM: warp-level mma.sync m16n8k8 TF32 with the 3xTF32 split
// (x = hi + lo, both TF32; acc += a_lo b_hi + a_hi b_lo + a_hi b_hi), which keeps fp32-level accuracy (~2^-21 per
// product) at 3 MMAs per tile.  Measured mma.sync rate on B200 (tests/prim_bench.py): 811 FLOP/clk/SM for TF32 = 3.2x
// the FFMA rate, so the split GEMM has ~1.06x the FFMA peak.  MEASURED (config 2, PINN step): FFMA engine 32.8 ms, 3xTF32
// 32.5 ms, plain TF32 25.7 ms with loss errors up to 1.3e-3 -> the FFMA engine stays the default (fp32 like the
// reference); these variants build with DMIP_TILE=MMA3 / DMIP_TILE=TF32X1 (csrc/build.sh) for experiments.
// Orientation: the WEIGHT slab is the A operand (M = output features, row stride N + 8), the 32 activation rows are B
// (four n-tiles of 8): a warp owns 2 R features x 32 rows; C fragments store as float2 along the row index.
__device__ __forceinline__ uint32_t to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

template <int R, bool kSplit>
__device__ void tile_gemm_mma(const float* in, float* out, const float* __restrict__ Wt, int K, float* wbuf) {
  constexpr int N = 64 * R;              // 512 or 256
  constexpr int kMT = R / 4;             // m-tiles (16 features) per warp: 2 or 1
  constexpr int kLdW = N + kSlabPad;
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int g = lane >> 2, t4 = lane & 3;
  const int n0 = warp * (16 * kMT);
  float acc[kMT][4][4];
#pragma unroll
  for (int m = 0; m < kMT; ++m)
#pragma unroll
    for (int n = 0; n < 4; ++n)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[m][n][e] = 0.f;
  const int n_slabs = K / kSlabK;
  constexpr int kChunksRow = N / 4;                 // 16-byte chunks per slab row
  constexpr int kChunks = kSlabK * kChunksRow;
  auto issue = [&](int s) {
    const float* src = Wt + static_cast<size_t>(s) * kSlabK * N;
    float* dst = wbuf + (s & 1) * kSlabK * kLdW;
    for (int c = t; c < kChunks; c += kThreadsL) {
      const int row = c / kChunksRow, col = c - row * kChunksRow;
      cp_async16(dst + row * kLdW + col * 4, src + c * 4);
    }
    cp_async_commit();
  };
  issue(0);
  for (int s = 0; s < n_slabs; ++s) {
    if (s + 1 < n_slabs) {
      issue(s + 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const float* w = wbuf + (s & 1) * kSlabK * kLdW + n0 + g;
    const float* a = in + s * kSlabK * kLd + g;
#pragma unroll
    for (int kk = 0; kk < kSlabK; kk += 8) {
      uint32_t bh[4][2], bl[4][2];
#pragma unroll
      for (int n = 0; n < 4; ++n)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const float x = a[(kk + t4 + 4 * e) * kLd + n * 8];
          bh[n][e] = to_tf32(x);
          if (kSplit) bl[n][e] = to_tf32(x - __uint_as_float(bh[n][e]));
        }
#pragma unroll
      for (int m = 0; m < kMT; ++m) {
        uint32_t ah[4], al[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float x = w[(kk + t4 + 4 * (e >> 1)) * kLdW + m * 16 + 8 * (e & 1)];
          ah[e] = to_tf32(x);
          if (kSplit) al[e] = to_tf32(x - __uint_as_float(ah[e]));
        }
#pragma unroll
        for (int n = 0; n < 4; ++n) {
          if (kSplit) {
            mma_tf32(acc[m][n], al, bh[n][0], bh[n][1]);
            mma_tf32(acc[m][n], ah, bl[n][0], bl[n][1]);
          }
          mma_tf32(acc[m][n], ah, bh[n][0], bh[n][1]);
        }
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int m = 0; m < kMT; ++m)
#pragma unroll
    for (int n = 0; n < 4; ++n) {
      float* o = out + (n0 + m * 16 + g) * kLd + n * 8 + 2 * t4;
      *reinterpret_cast<float2*>(o) = make_float2(acc[m][n][0], acc[m][n][1]);
      *reinterpret_cast<float2*>(o + 8 * kLd) = make_float2(acc[m][n][2], acc[m][n][3]);
    }
  __syncthreads();
}

// out[n*kLd + r] = sum_k in[k*kLd + r] * Wt[k*N + n]: staged path for the big square layers, skinny path for few
// outputs behind a long contraction, direct path otherwise
__device__ void tile_gemm(const float* in, float* out, const float* __restrict__ Wt, int K, int N, float* wbuf) {
  if (N <= 32 && K >= 64) { tile_gemm_skinny(in, out, Wt, K, N); return; }
  if ((K % kSlabK) == 0 && K >= 64 && (reinterpret_cast<uintptr_t>(Wt) & 15) == 0) {
#if defined(DMIP_TILE_TF32X1)      // experiment: plain TF32 (errors up to 1.3e-3 on the loss fixtures, PINN step 25.7 ms)
    if (N == 512) { tile_gemm_mma<8, false>(in, out, Wt, K, wbuf); return; }
    if (N == 256) { tile_gemm_mma<4, false>(in, out, Wt, K, wbuf); return; }
#elif defined(DMIP_TILE_MMA3)      // experiment: 3xTF32 (fp32-level accuracy, PINN step 32.5 ms = the FFMA engine's)
    if (N == 512) { tile_gemm_mma<8, true>(in, out, Wt, K, wbuf); return; }
    if (N == 256) { tile_gemm_mma<4, true>(in, out, Wt, K, wbuf); return; }
#else
    if (N == 512) { tile_gemm_staged<8>(in, out, Wt, K, wbuf); return; }
    if (N == 256) { tile_gemm_staged<4>(in, out, Wt, K, wbuf); return; }
#endif
  }
  tile_gemm_direct(in, out, Wt, K, N);
}


__global__ void k_transpose_l(const float* __restrict__ W, float* __restrict__ Wt, int rows, int cols) {
  __shared__ float tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < rows && c < cols) ? W[static_cast<size_t>(r) * cols + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (r < rows && c < cols) Wt[static_cast<size_t>(c) * rows + r] = tile[threadIdx.x][i];
  }
}


inline size_t align_up(size_t v) { return (v + 255) & ~size_t(255); }

// ---- a DmipMlp on this engine.  Its weights are used transposed ([k][n]) from the caller's workspace, every layer at a
// 256-byte boundary so that tile_gemm's staged path (16-byte cp.async) applies whenever the layer shape allows it.

// Refuses a net the engine cannot run.  want_in: the in_dim the caller's inputs give (net.in_dim where it has none).
inline int tile_net_check(const DmipMlp& net, int want_in, const char* what) {
  DMIP_REQUIRE(net.n_layers >= 2 && net.n_layers <= DMIP_MAX_LAYERS, "%s: n_layers %d out of range (2..%d)", what,
               net.n_layers, DMIP_MAX_LAYERS);
  DMIP_REQUIRE(net.in_dim == want_in && net.in_dim >= 1 && net.in_dim <= kMaxW, "%s: in_dim must be %d (1..%d), got %d",
               what, want_in, kMaxW, net.in_dim);
  for (int l = 0; l < net.n_layers; ++l) {
    DMIP_REQUIRE(net.width[l] >= 1 && net.width[l] <= kMaxW, "%s: bad width: layer %d width %d out of range (1..%d)", what,
                 l, net.width[l], kMaxW);
    DMIP_REQUIRE(net.W[l] && net.b[l], "%s: layer %d has a NULL pointer", what, l);
  }
  DMIP_REQUIRE(net.width[net.n_layers - 1] == net.out_dim, "%s: last layer width %d != out_dim %d", what,
               net.width[net.n_layers - 1], net.out_dim);
  return DMIP_OK;
}

// Workspace bytes of the transposed weights.  Workspace queries come before the check, so a bad descriptor is sized
// without reading past width[DMIP_MAX_LAYERS - 1].
inline size_t tile_net_bytes(const DmipMlp& net) {
  size_t bytes = 0;
  int k = net.in_dim;
  for (int l = 0; l < net.n_layers && l < DMIP_MAX_LAYERS; ++l) {
    if (k < 0 || net.width[l] < 0) return 0;
    bytes += align_up(sizeof(float) * k * net.width[l]);
    k = net.width[l];
  }
  return bytes;
}

// Transposes the weights into ws (tile_net_bytes of it) and fills the net fields every FFMA device struct carries.
template <class Dev>
int tile_net_stage(const DmipMlp& net, void* ws, Dev* d, cudaStream_t s) {
  d->n_layers = net.n_layers;
  d->in_dim = net.in_dim;
  d->out_dim = net.out_dim;
  uint8_t* p = static_cast<uint8_t*>(ws);
  int k = net.in_dim;
  for (int l = 0; l < net.n_layers; ++l) {
    const int n = net.width[l];
    float* wt = reinterpret_cast<float*>(p);
    d->width[l] = n;
    d->b[l] = net.b[l];
    d->Wt[l] = wt;
    dim3 grid(ceil_div(k, 32), ceil_div(n, 32)), block(32, 8);
    k_transpose_l<<<grid, block, 0, s>>>(net.W[l], wt, n, k);
    DMIP_CHECK_CUDA(cudaGetLastError());
    count_launch();
    p += align_up(sizeof(float) * k * n);
    k = n;
  }
  return DMIP_OK;
}

}  // namespace
}  // namespace dmip
