// dmip_mmd_test.cu — permutation two-sample test on the unbiased MMD^2 (Gretton et al. 2012, JMLR 13, eq. 3 and §5):
// the statistic of the observed split and of up to DMIP_MMD_TEST_MAX_PERM relabelings of the pooled points, from ONE
// pass over the pooled kernel matrix.
//
// Pooled points z = [x; y] (N = n + m), mixture kernel k(a, c) = sum_b exp(-|a - c|^2 / (2 sigma_b^2)) with K_ii = 0.
// For a labeling u in {0,1}^N with n ones, A = u'Ku, B = u'K1, T = 1'K1 give Sxx = A, Sxy = B - A, Syy = T - 2B + A and
// MMD^2_u = Sxx / (n(n-1)) + Syy / (m(m-1)) - 2 Sxy / (nm).  With U = [u_0 | u_1 .. u_P | 1 | 0 pad] (u_0: x first),
// R = K U holds every A_p = sum_i u_ip R_ip, B_p = sum_i u_ip R_i,ones and T = sum_i R_i,ones.
//
// k_mmd_test: one CTA per (observation, 128-row tile I) walks the 64-column tiles J of its observation.
//   warps 0-3 (one pooled row per thread): the kernel tile K[I, J] in packed fp32 (differences, ex2 per bandwidth as
//             k_mmd), summed over bandwidths, rounded to the fixed point q = rint(k 2047 / n_bw) = 128 hi + lo and
//             written as the u8 A operand row [hi(64) | lo(64)] (K-major SWIZZLE_128B, 16 KB);
//   warps 4-7: the label bits of tile J + 1 expanded into the u8 B operand rows [128 u | u] (nc x 128 bytes,
//             nc = round_up(P + 2, 16)) and its 64 column points staged for the compute warps;
//   one elected lane of warp 0: four tcgen05.mma kind::i8 (M = 128, N = nc, K = 32) into an s32 TMEM accumulator,
//             committed to the stage's mbarrier.
// The products and their sums are exact integers: the only rounding is that of each kernel value to 1/2047 of n_bw.
// (An f16 A operand with the fp32 accumulator was measured first: the tensor core's accumulation error grows with the
// number of K steps and differs between the contiguous observed split and the scattered permutations, so at
// n = m = 2^16 the observed statistic sat ~100 null standard deviations off; DESIGN.md §3 "MMD permutation test".)
// A and B are double-buffered, so the ex2 work of tile J + 1 runs under the MMAs of tile J (one __syncthreads per tile).
// Epilogue: tcgen05.ld of the 128 x nc s32 rows, each weighted by the row's own label bit, converted to fp64 (exact:
// every sum stays below 2^53) and reduced over the warp (butterfly, fixed order) and over the four warps in warp order
// into workspace slot (o, I).  k_mmd_test_finish (one block per observation) sums the slots in tile order, forms the statistics, checks
// every label row's popcount and counts exceedances.  Two launches per call, bit-identical from run to run.
#include <float.h>
#include <math.h>
#include <math_constants.h>

#include "dmip_common.h"
#include "dmip_ptx.cuh"

namespace dmip {

namespace {

constexpr int kThreads = 256;
constexpr int kRows = 128;                   // pooled rows per CTA (MMA M)
constexpr int kCols = 64;                    // pooled columns per tile (MMA K: one 128-byte f16 swizzle row)
constexpr int kMaxNc = 256;                  // accumulator columns: P + 2 rounded up to 16
constexpr uint32_t kABytes = kRows * 128;    // 16 KB
constexpr uint32_t kBBytes = kMaxNc * 128;   // 32 KB
constexpr uint32_t kOffB = 2 * kABytes;
constexpr uint32_t kOffCols = kOffB + 2 * kBBytes;
constexpr uint32_t kColsBytes = kCols * 16 * 4;                   // 64 points x 16 dims fp32, per stage
constexpr uint32_t kOffBars = kOffCols + 2 * kColsBytes;
constexpr uint32_t kSmem = kOffBars + 64 + 1024;                    // + alignment slack of the dynamic window
// Fixed-point kernel values q = rint(k 2047 / n_bw) <= 2047: a row sum of N <= 2^20 of them stays below 2^31, so the
// s32 tensor-memory accumulator holds R exactly (no accumulation rounding at any N), and every fp64 sum of them is exact.
constexpr uint32_t kQMax = 2047;

// D[tmem] (+)= A[smem] * B[smem]^T, kind::i8 (u8 x u8 -> s32)      (issued by ONE thread)
__device__ __forceinline__ void umma_ss_i8(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// instruction descriptor, kind::i8: D = s32 (2 << 4), A = B = u8 (format 0), both K-major
__host__ __device__ constexpr uint32_t umma_idesc_u8(uint32_t M, uint32_t N) { return (2u << 4) | ((N >> 3) << 17) | ((M >> 4) << 24); }

struct TestParams {
  const float* x;            // (n_obs, n, dim)
  const float* y;            // (n_obs, m, dim)
  const uint32_t* labels;    // (n_obs, P, W)
  long long n, m, N;
  int dim, P, nc, nb;
  long long W;               // label words per row: ceil(N / 32)
  long long tiles;           // 128-row tiles per observation
  long long jtiles;          // 64-column tiles per observation
  float scale;               // s = sqrt(log2(e) / (2 sigma_0^2))
  float ratio[DMIP_MMD_MAX_BW];
  float qscale;              // kQMax / n_bw: fixed-point units per kernel value
  double* partial;           // (n_obs, tiles, 2, kMaxNc)
};

__device__ __forceinline__ float ex2_neg(float t) {   // 2^-t on the MUFU
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(-t));
  return r;
}

__device__ __forceinline__ const float* point(const TestParams& P, long long o, long long j) {
  return j < P.n ? P.x + (o * P.n + j) * P.dim : P.y + (o * P.m + (j - P.n)) * P.dim;
}

// label word w of accumulator column c for observation o: column 0 is the observed split (x first), 1..P the caller's
// rows, P + 1 the ones column, the rest zero; bits of points >= N are cleared
__device__ __forceinline__ uint32_t label_word(const TestParams& P, long long o, int c, long long w) {
  if (w >= P.W) return 0u;
  const long long b0 = w * 32;
  const uint32_t valid = P.N - b0 >= 32 ? 0xffffffffu : (1u << (P.N - b0)) - 1u;
  uint32_t v;
  if (c == 0) {
    v = P.n - b0 >= 32 ? 0xffffffffu : P.n <= b0 ? 0u : (1u << (P.n - b0)) - 1u;
  } else if (c <= P.P) {
    v = __ldg(P.labels + (o * P.P + (c - 1)) * P.W + w);
  } else {
    v = c == P.P + 1 ? 0xffffffffu : 0u;
  }
  return v & valid;
}

// Byte offset of byte b (0..127) of row `row` in a K-major SWIZZLE_128B u8 tile (the layout of sw128_offset, in bytes)
__device__ __forceinline__ uint32_t sw128_byte(uint32_t row, uint32_t b) {
  return (row >> 3) * 1024u + (row & 7u) * 128u + ((((b >> 4) ^ (row & 7u))) << 4) + (b & 15u);
}

// B operand of column tile J (rows = accumulator columns; bytes [128 u_j | u_j] for the tile's 64 points j, matching
// the A row [hi | lo]) and the tile's column points as (-s c_j, -s c_j+1) pairs; executed by the 128 threads of warps 4-7
template <int DP>
__device__ __forceinline__ void stage_columns(const TestParams& P, long long o, long long J, uint8_t* b, float2* cols,
                                              int t) {
  for (int e = t; e < P.nc * 2; e += 128) {
    const int c = e >> 1, h = e & 1;
    const uint32_t w = label_word(P, o, c, J * 2 + h);
#pragma unroll
    for (int q = 0; q < 2; ++q) {                             // points h * 32 + 16 q .. + 15
      uint32_t v[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint32_t nib = (w >> (16 * q + 4 * k)) & 15u;   // one byte 0 / 1 per point
        v[k] = (nib & 1u) | ((nib & 2u) << 7) | ((nib & 4u) << 14) | ((nib & 8u) << 21);
      }
      const int col = h * 32 + q * 16;
      *reinterpret_cast<uint4*>(b + sw128_byte(c, col)) = make_uint4(v[0] << 7, v[1] << 7, v[2] << 7, v[3] << 7);
      *reinterpret_cast<uint4*>(b + sw128_byte(c, 64 + col)) = make_uint4(v[0], v[1], v[2], v[3]);
    }
  }
  for (int e = t; e < kCols * DP; e += 128) {
    const int j = e / DP, k = e - j * DP;
    const long long jg = J * kCols + j;
    const float v = (jg < P.N && k < P.dim) ? -__ldg(point(P, o, jg) + k) * P.scale : 0.f;
    reinterpret_cast<float*>(cols)[((j >> 1) * DP + k) * 2 + (j & 1)] = v;
  }
}

// row `gi` of kernel tile J -> the A operand row [hi(64) | lo(64)] of the fixed-point kernel values q = hi 128 + lo;
// R holds the row's scaled coordinates as (v, v) pairs
template <int DP>
__device__ __forceinline__ void kernel_row(const TestParams& P, const unsigned long long (&R)[DP],
                                           const unsigned long long* rb, long long gi, long long J, int row,
                                           const float2* cols, uint8_t* a) {
  const long long j0 = J * kCols;
#pragma unroll 1
  for (int q = 0; q < 4; ++q) {                               // columns j0 + 16 q .. + 15
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      const int pr = q * 8 + w;                               // columns j0 + 2 pr, j0 + 2 pr + 1
      unsigned long long dist = 0ull;
#pragma unroll
      for (int k = 0; k < DP; ++k) {
        const float2 c = cols[pr * DP + k];
        const unsigned long long df = f32x2_add(R[k], f32x2_pack(c.x, c.y));
        dist = k == 0 ? f32x2_mul(df, df) : f32x2_fma(df, df, dist);
      }
      unsigned long long acc = 0ull;
#pragma unroll
      for (int bw = 0; bw < DMIP_MMD_MAX_BW; ++bw) {
        if (bw < P.nb) {
          const unsigned long long t = f32x2_mul(dist, rb[bw]);
          float t0, t1;
          f32x2_unpack(t, t0, t1);
          acc = f32x2_add(acc, f32x2_pack(ex2_neg(t0), ex2_neg(t1)));
        }
      }
      float k0, k1;
      f32x2_unpack(acc, k0, k1);
      const long long jg = j0 + 2 * pr;
      if (jg == gi || jg >= P.N) k0 = 0.f;                    // the diagonal is masked explicitly, not by distance 0
      if (jg + 1 == gi || jg + 1 >= P.N) k1 = 0.f;
      const uint32_t q0 = min(static_cast<uint32_t>(__float2int_rn(k0 * P.qscale)), kQMax);
      const uint32_t q1 = min(static_cast<uint32_t>(__float2int_rn(k1 * P.qscale)), kQMax);
      const uint32_t sh = 16u * (w & 1);                       // bytes 2 (w & 1), 2 (w & 1) + 1 of word w / 2
      const uint32_t h2 = ((q0 >> 7) | ((q1 >> 7) << 8)) << sh, l2 = ((q0 & 127u) | ((q1 & 127u) << 8)) << sh;
      if (w & 1) {
        hi[w >> 1] |= h2;
        lo[w >> 1] |= l2;
      } else {
        hi[w >> 1] = h2;
        lo[w >> 1] = l2;
      }
    }
    *reinterpret_cast<uint4*>(a + sw128_byte(row, q * 16)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(a + sw128_byte(row, 64 + q * 16)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}

// column sums of v[32] over the warp: afterwards lane L holds column L in v[0] (fixed summation tree)
__device__ __forceinline__ double warp_column_sums(double (&v)[32], int lane) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    const bool up = (lane & off) != 0;
#pragma unroll
    for (int q = 0; q < off; ++q) {
      const double send = up ? v[q] : v[q + off];
      const double keep = up ? v[q + off] : v[q];
      v[q] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  return v[0];
}

template <int DP>
__global__ void __launch_bounds__(kThreads, 2) k_mmd_test(const __grid_constant__ TestParams P) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // SWIZZLE_128B operands: 1024 B aligned
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kOffBars);   // [0], [1]: MMA of stage done
  uint32_t* holder = reinterpret_cast<uint32_t*>(bars + 2);
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const long long o = blockIdx.x / P.tiles, I = blockIdx.x - o * P.tiles;
  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc<kMaxNc>(holder);
  if (warp >= 4) stage_columns<DP>(P, o, 0, smem + kOffB, reinterpret_cast<float2*>(smem + kOffCols), tid - 128);
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *holder;

  const long long gi = I * kRows + tid;                          // this thread's pooled row (warps 0-3)
  unsigned long long R[DP];
  unsigned long long rb[DMIP_MMD_MAX_BW];
  if (warp < 4) {
#pragma unroll
    for (int k = 0; k < DP; ++k) {
      const float v = (gi < P.N && k < P.dim) ? __ldg(point(P, o, gi) + k) * P.scale : 0.f;
      R[k] = f32x2_pack(v, v);
    }
#pragma unroll
    for (int b = 0; b < DMIP_MMD_MAX_BW; ++b) rb[b] = f32x2_pack(P.ratio[b], P.ratio[b]);
  }
  const uint32_t idesc = umma_idesc_u8(kRows, static_cast<uint32_t>(P.nc));
  for (long long J = 0; J < P.jtiles; ++J) {
    const int s = static_cast<int>(J & 1);
    if (warp < 4) {
      if (J >= 2) mbar_wait(&bars[s], static_cast<uint32_t>(((J - 2) >> 1) & 1), 0x300 + s);
      kernel_row<DP>(P, R, rb, gi, J, tid, reinterpret_cast<const float2*>(smem + kOffCols + s * kColsBytes),
                     smem + s * kABytes);
    } else if (J + 1 < P.jtiles) {
      const int s1 = s ^ 1;
      if (J >= 1) mbar_wait(&bars[s1], static_cast<uint32_t>(((J - 1) >> 1) & 1), 0x310 + s1);
      stage_columns<DP>(P, o, J + 1, smem + kOffB + s1 * kBBytes,
                        reinterpret_cast<float2*>(smem + kOffCols + s1 * kColsBytes), tid - 128);
    }
    fence_proxy_async_smem();
    __syncthreads();
    if (warp == 0) {
      tc_fence_after();
      if (elect_one()) {
        const uint32_t a0 = smem_u32(smem + s * kABytes), b0 = smem_u32(smem + kOffB + s * kBBytes);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)                          // K = 32 bytes per instruction
          umma_ss_i8(tmem, umma_smem_desc_sw128(a0 + 32 * kk), umma_smem_desc_sw128(b0 + 32 * kk), idesc,
                  (J > 0 || kk > 0) ? 1u : 0u);
        tc_commit(&bars[s]);
      }
      __syncwarp();
    }
  }

  // ---- epilogue: weight the accumulator rows by their own label bits, fp64 column sums in a fixed order
  double* red = reinterpret_cast<double*>(smem);                  // [2][4 warps][kMaxNc]: the A stages are free now
  if (warp < 4) {
    const long long last = P.jtiles - 1;
    mbar_wait(&bars[last & 1], static_cast<uint32_t>((last >> 1) & 1), 0x320);
    tc_fence_after();
    const uint32_t trow = tmem + (static_cast<uint32_t>(warp * 32) << 16);
    const bool valid = gi < P.N;
    const long long wrow = (I * kRows + warp * 32) >> 5;          // the warp's 32 rows share one label word per column
    const int ones_col = P.P + 1;
    uint32_t ones;
    {
      uint32_t r[32];
      tmem_ld32(trow + static_cast<uint32_t>(ones_col & ~31), r);
      tc_wait_ld();
      ones = 0u;
#pragma unroll
      for (int q = 0; q < 32; ++q)
        if (q == (ones_col & 31)) ones = r[q];
    }
    const double ones_d = valid ? static_cast<double>(static_cast<int>(ones)) : 0.0;
    for (int ch = 0; ch * 32 < P.nc; ++ch) {
      uint32_t bits = 0u;
      for (int q = 0; q < 32; ++q) bits |= ((label_word(P, o, ch * 32 + q, wrow) >> lane) & 1u) << q;
      if (!valid) bits = 0u;
      uint32_t r[32];
      tmem_ld32(trow + static_cast<uint32_t>(ch * 32), r);
      tc_wait_ld();
      double v[32];
#pragma unroll
      for (int q = 0; q < 32; ++q) v[q] = (bits >> q) & 1u ? static_cast<double>(static_cast<int>(r[q])) : 0.0;
      red[(0 * 4 + warp) * kMaxNc + ch * 32 + lane] = warp_column_sums(v, lane);
#pragma unroll
      for (int q = 0; q < 32; ++q) v[q] = (bits >> q) & 1u ? ones_d : 0.0;
      red[(1 * 4 + warp) * kMaxNc + ch * 32 + lane] = warp_column_sums(v, lane);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc<kMaxNc>(tmem);
  }
  double* slot = P.partial + (o * P.tiles + I) * 2 * kMaxNc;
  for (int e = tid; e < 2 * kMaxNc; e += kThreads) {
    const int h = e / kMaxNc, c = e - h * kMaxNc;
    double s = 0.0;
    if (c < P.nc)
      for (int w = 0; w < 4; ++w) s += red[(h * 4 + w) * kMaxNc + c];
    slot[e] = s;
  }
}

// One block per observation, thread c = accumulator column 0..P: the slots in tile order, the statistic, the popcount of
// the label row, and the exceedance count over the block.
__global__ void __launch_bounds__(kMaxNc) k_mmd_test_finish(const TestParams P, double* out, double* p_value) {
  const long long o = blockIdx.x;
  const int c = threadIdx.x;
  __shared__ double stat0;
  double stat = 0.0;
  bool bad = false;
  if (c <= P.P) {
    const double* base = P.partial + o * P.tiles * 2 * kMaxNc;
    double A = 0.0, B = 0.0, T = 0.0;
    for (long long I = 0; I < P.tiles; ++I) {
      const double* slot = base + I * 2 * kMaxNc;
      A += slot[c];
      B += slot[kMaxNc + c];
      T += slot[P.P + 1];
    }
    if (c > 0) {
      long long pop = 0;
      for (long long w = 0; w < P.W; ++w) pop += __popc(label_word(P, o, c, w));
      bad = pop != P.n;
    }
    const double n = static_cast<double>(P.n), m = static_cast<double>(P.m);
    const double sxx = A, sxy = B - A, syy = T - 2.0 * B + A;
    stat = bad ? CUDART_NAN : (sxx / (n * (n - 1.0)) + syy / (m * (m - 1.0)) - 2.0 * sxy / (n * m)) / P.qscale;
    out[o * (P.P + 1) + c] = stat;
    if (c == 0) stat0 = stat;
  }
  __syncthreads();
  const int exceed = __syncthreads_count(c >= 1 && c <= P.P && stat >= stat0);
  const int any_bad = __syncthreads_or(bad);
  if (c == 0 && p_value) p_value[o] = any_bad ? CUDART_NAN : (1.0 + exceed) / (P.P + 1.0);
}

template <int DP>
int run(const TestParams& P, long long grid, cudaStream_t s) {
  static bool ready[64] = {};
  int dev = 0;
  DMIP_CHECK_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || !ready[dev]) {
    DMIP_CHECK_CUDA(cudaFuncSetAttribute(k_mmd_test<DP>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));
    if (dev >= 0 && dev < 64) ready[dev] = true;
  }
  k_mmd_test<DP><<<static_cast<unsigned>(grid), kThreads, kSmem, s>>>(P);
  DMIP_CHECK_CUDA(cudaGetLastError());
  return DMIP_OK;
}

long long row_tiles(long long N) { return (N + kRows - 1) / kRows; }

}  // namespace

size_t mmd_test_workspace(const DmipMmdTest* d) {
  if (!d || d->n_obs < 1 || d->n < 2 || d->m < 2 || d->n + d->m > DMIP_MMD_TEST_MAX_POINTS) return 0;
  return static_cast<size_t>(d->n_obs) * static_cast<size_t>(row_tiles(d->n + d->m)) * 2 * kMaxNc * sizeof(double);
}

int launch_mmd_test(const DmipMmdTest* d, cudaStream_t s) {
  DMIP_REQUIRE(d->dim >= 1 && d->dim <= DMIP_MMD_MAX_DIM, "MMD test dimension must be 1..%d (got %d)", DMIP_MMD_MAX_DIM,
               d->dim);
  DMIP_REQUIRE(d->n_obs >= 1, "MMD test needs n_obs >= 1 (got %d)", d->n_obs);
  DMIP_REQUIRE(d->n >= 2 && d->m >= 2, "MMD test needs at least 2 samples per set (n = %lld, m = %lld)",
               static_cast<long long>(d->n), static_cast<long long>(d->m));
  DMIP_REQUIRE(d->n + d->m <= DMIP_MMD_TEST_MAX_POINTS, "MMD test needs n + m <= %d pooled points (got %lld)",
               DMIP_MMD_TEST_MAX_POINTS, static_cast<long long>(d->n + d->m));
  DMIP_REQUIRE(d->n_bw >= 1 && d->n_bw <= DMIP_MMD_MAX_BW, "MMD test needs 1..%d bandwidths (got %d)", DMIP_MMD_MAX_BW,
               d->n_bw);
  for (int b = 0; b < d->n_bw; ++b)
    DMIP_REQUIRE(d->sigma[b] > 0.f && isfinite(d->sigma[b]), "bandwidth %d must be positive and finite (got %g)", b,
                 static_cast<double>(d->sigma[b]));
  DMIP_REQUIRE(d->n_perm >= 1 && d->n_perm <= DMIP_MMD_TEST_MAX_PERM, "MMD test needs 1..%d permutations (got %d)",
               DMIP_MMD_TEST_MAX_PERM, d->n_perm);
  DMIP_REQUIRE(d->x && d->y && d->labels && d->out, "x / y / labels / out is NULL");
  DMIP_REQUIRE((reinterpret_cast<uintptr_t>(d->labels) & 3) == 0, "labels must be 4-byte aligned");
  const long long N = d->n + d->m, tiles = row_tiles(N);
  DMIP_REQUIRE(static_cast<long long>(d->n_obs) * tiles < (1LL << 31), "too many observations for one call (%d)",
               d->n_obs);
  if (!d->workspace || d->workspace_bytes < mmd_test_workspace(d)) {
    set_error("workspace too small: need %zu bytes", mmd_test_workspace(d));
    return DMIP_EWORKSPACE;
  }
  DMIP_REQUIRE((reinterpret_cast<uintptr_t>(d->workspace) & 7) == 0, "workspace must be 8-byte aligned");

  TestParams P = {};
  P.x = d->x;
  P.y = d->y;
  P.labels = d->labels;
  P.n = d->n;
  P.m = d->m;
  P.N = N;
  P.dim = d->dim;
  P.P = d->n_perm;
  P.nc = (d->n_perm + 2 + 15) / 16 * 16;
  P.nb = d->n_bw;
  P.W = (N + 31) / 32;
  P.tiles = tiles;
  P.jtiles = (N + kCols - 1) / kCols;
  const double s0 = d->sigma[0];
  P.scale = static_cast<float>(sqrt(1.4426950408889634 / (2.0 * s0 * s0)));
  for (int b = 0; b < d->n_bw; ++b) {
    const double r = (s0 / d->sigma[b]) * (s0 / d->sigma[b]);
    P.ratio[b] = static_cast<float>(r < FLT_MAX ? r : FLT_MAX);
  }
  P.qscale = static_cast<float>(kQMax) / static_cast<float>(d->n_bw);
  P.partial = static_cast<double*>(d->workspace);

  const long long grid = d->n_obs * tiles;
  const int dp = d->dim <= 4 ? d->dim : d->dim <= 8 ? 8 : 16;
  int rc;
  switch (dp) {
    case 1: rc = run<1>(P, grid, s); break;
    case 2: rc = run<2>(P, grid, s); break;
    case 3: rc = run<3>(P, grid, s); break;
    case 4: rc = run<4>(P, grid, s); break;
    case 8: rc = run<8>(P, grid, s); break;
    default: rc = run<16>(P, grid, s); break;
  }
  if (rc) return rc;
  count_launch();
  k_mmd_test_finish<<<static_cast<unsigned>(d->n_obs), kMaxNc, 0, s>>>(P, d->out, d->p_value);
  DMIP_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return DMIP_OK;
}

}  // namespace dmip
