// dmip_ksd.cu — kernel Stein discrepancy of a sample set against a target known through its score (Liu, Lee & Jordan
// 2016; Chwialkowski, Strathmann & Gretton 2016), for up to DMIP_MMD_MAX_BW kernel scales at once.  No reference
// counterpart.  It needs no ground-truth samples: only the points x_i and the target's score s_i = grad log p(x_i).
//
// With delta = x_i - x_j, r^2 = |delta|^2 and a = (s_i - s_j).delta + d, the Stein kernel
// u(x, x') = s.s' k + s.grad_x' k + s'.grad_x k + tr grad_x grad_x' k is, per scale,
//   IMQ (c, beta = -1/2):  k = (c^2 + r^2)^(-1/2),   u_ij = k s_i.s_j + k^3 a - 3 r^2 k^5,     u_ii = |s_i|^2 / c + d / c^3
//   Gaussian (sigma):      k = exp(-r^2 / (2 s^2)),  u_ij = k [s_i.s_j + a / s^2 - r^2 / s^4], u_ii = |s_i|^2 + d / s^2
// and per observation KSD^2_U = sum_{i != j} u_ij / (n (n - 1)), KSD^2_V = sum_{i, j} u_ij / n^2 (oracle/ksd.py).
//
// Arithmetic: a thread holds RPT rows as packed pairs (two rows per 64-bit register); the columns stream through shared
// memory as duplicated pairs (-x_j, -x_j) and (s_j, s_j).  Per two pairs and dimension: one FADD2 (delta), one FFMA2 (r^2),
// one FFMA2 (s_i.s_j), one FADD2 (s_i - s_j) and one FFMA2 (a; the first dimension starts it at d), 5d FP32 operations
// per pair.  Per scale and two pairs: IMQ one FADD2 (c^2 + r^2), two MUFU.RSQ, one FMUL2 (k^2) and three FFMA2
// (k^2 (a - 3 r^2 k^2), + s_i.s_j, k (...) + acc) after one FMUL2 (-3 r^2) per pair; Gaussian one FMUL2, two MUFU.EX2 and
// three FFMA2.  At d >= 2 the FP32 issue slots bind, not the MUFU (DESIGN.md §3 "Evaluation metrics").
//
// Work: per observation the tiles I <= J of the T x T tiling of the n x n square, one work unit each, numbered
// observation-major; every CTA of the persistent grid takes one contiguous range of units.  Off-diagonal tiles count
// twice (u is symmetric); on diagonal tiles the pair i = j gets k = 0 in the pair loop and its closed form u_ii goes, in
// fp64, to a second sum that only KSD^2_V uses.  Per-row fp32 sums cover at most T columns and are folded into fp64
// after every tile; slots, CTA order and the finish kernel are k_mmd's (dmip_pairs.cuh).  Two launches per call,
// bit-identical from run to run on one device.  A non-finite score gives a NaN result: nothing is masked.
#include <float.h>
#include <math.h>
#include <string.h>

#include "dmip_common.h"
#include "dmip_pairs.cuh"
#include "dmip_ptx.cuh"

namespace dmip {

namespace {

using pairs::flush_group;
using pairs::tri_decode;

constexpr int kThreads = 256;
constexpr int kUnroll = 4;         // column loop unroll; the remainder of a chunk runs one column at a time
constexpr int kMaxGrid = 1024;     // bounds the workspace independently of the device

// columns staged in shared memory at a time: 2 DP packed values each, at most 32 KB
__host__ __device__ constexpr int chunk_cols(int dp) { return dp == 16 ? 128 : kThreads; }

// rows held per thread (the tile edge is 256 x this) and CTAs per SM: as many rows as fit 128 registers without spilling
// at two CTAs per SM; where even two rows spill there (d = 16, and d = 4 with 8 scales), one CTA per SM with 255 registers
constexpr int rows_per_thread(int dp, int ns) {
  return dp <= 2 ? (ns <= 4 ? 8 : 4) : dp <= 4 ? (ns == 1 ? 8 : ns <= 3 ? 4 : 2) : 2;
}
__host__ __device__ constexpr int ctas_per_sm(int dp, int ns) { return dp == 16 || (dp == 4 && ns == 8) ? 1 : 2; }

struct KsdParams {
  const float* x;                   // (n_obs, n, dim)
  const float* s;                   // (n_obs, n, dim)
  long long n;
  int dim;
  // per scale, as duplicated fp32 pairs (packed operands straight from the parameter bank)
  unsigned long long c2[DMIP_MMD_MAX_BW];     // IMQ: c^2;  Gaussian: log2(e) / (2 sigma^2)
  unsigned long long inv2[DMIP_MMD_MAX_BW];   // Gaussian: 1 / sigma^2
  unsigned long long ninv4[DMIP_MMD_MAX_BW];  // Gaussian: -1 / sigma^4
  double diag_a[DMIP_MMD_MAX_BW];   // u_ii = diag_a |s_i|^2 + diag_b
  double diag_b[DMIP_MMD_MAX_BW];
  long long t;                      // tiles along one side
  long long u_obs, u_total;         // units of one observation, of the call
  double* partial;                  // (kMaxGrid + n_obs) x 2 n_scales fp64 slots: {off-diagonal sums, diagonal sums}
};

__device__ __forceinline__ float ex2_neg(float t) {   // 2^-t on the MUFU
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(-t));
  return r;
}
__device__ __forceinline__ float rsqrt_mufu(float q) {   // one MUFU.RSQ
  float r;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(q));
  return r;
}
__device__ __forceinline__ unsigned long long f32x2_sub(unsigned long long a, unsigned long long b) {
  unsigned long long r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}

// One T x T tile of observation `o`: rows [I T, I T + T) against columns [J T, J T + T).
template <bool GAUSS, int DP, int NS, int RPT, bool DIAG>
__device__ __forceinline__ void tile(const KsdParams& P, const float* __restrict__ xo, const float* __restrict__ so,
                                     long long I, long long J, double w, double (&accd)[2 * NS],
                                     unsigned long long (*cs)[2 * DP]) {
  constexpr int T = kThreads * RPT, NP = RPT / 2, CH = chunk_cols(DP);
  const int tid = threadIdx.x;
  const int dim = P.dim;
  const long long n = P.n;
  unsigned long long X[NP][DP], S[NP][DP];
  bool valid[RPT];
#pragma unroll
  for (int p = 0; p < NP; ++p) {
    float v[2][DP], q[2][DP];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const long long i = I * T + static_cast<long long>(2 * p + h) * kThreads + tid;
      valid[2 * p + h] = i < n;
      double ss = 0.0;
#pragma unroll
      for (int k = 0; k < DP; ++k) {
        const bool in = i < n && (DP <= 4 || k < dim);
        v[h][k] = in ? __ldg(xo + i * dim + k) : 0.f;
        q[h][k] = in ? __ldg(so + i * dim + k) : 0.f;
        ss += static_cast<double>(q[h][k]) * static_cast<double>(q[h][k]);
      }
      if (DIAG && i < n)
#pragma unroll
        for (int b = 0; b < NS; ++b) accd[NS + b] += P.diag_a[b] * ss + P.diag_b[b];
    }
#pragma unroll
    for (int k = 0; k < DP; ++k) {
      X[p][k] = f32x2_pack(v[0][k], v[1][k]);
      S[p][k] = f32x2_pack(q[0][k], q[1][k]);
    }
  }
  const unsigned long long dd = f32x2_pack(static_cast<float>(dim), static_cast<float>(dim));
  const unsigned long long m3 = f32x2_pack(-3.f, -3.f);
  unsigned long long A[NP][NS];
#pragma unroll
  for (int p = 0; p < NP; ++p)
#pragma unroll
    for (int b = 0; b < NS; ++b) A[p][b] = 0ull;

  const long long c0 = J * T;
  const int ncol = static_cast<int>(n - c0 < T ? n - c0 : T);
  for (int ch = 0; ch < ncol; ch += CH) {
    const int cnt = ncol - ch < CH ? ncol - ch : CH;
    __syncthreads();                                   // the previous chunk's readers are done
    if (tid < cnt) {
      const long long j = c0 + ch + tid;
#pragma unroll
      for (int k = 0; k < DP; ++k) {
        const bool in = DP <= 4 || k < dim;
        const float xv = in ? -__ldg(xo + j * dim + k) : 0.f;
        const float sv = in ? __ldg(so + j * dim + k) : 0.f;
        cs[tid][k] = f32x2_pack(xv, xv);
        cs[tid][DP + k] = f32x2_pack(sv, sv);
      }
    }
    __syncthreads();
    // column c of the chunk against the thread's rows
    auto column = [&](int c) {
      unsigned long long Cx[DP], Cs[DP];
#pragma unroll
      for (int k = 0; k < DP; ++k) {
        Cx[k] = cs[c][k];
        Cs[k] = cs[c][DP + k];
      }
      const int rel = ch + c - tid;                    // DIAG: row slot h holds this column when rel == h * kThreads
#pragma unroll
      for (int p = 0; p < NP; ++p) {
        unsigned long long r2 = 0ull, ss = 0ull, a = 0ull;
#pragma unroll
        for (int k = 0; k < DP; ++k) {
          const unsigned long long df = f32x2_add(X[p][k], Cx[k]);
          const unsigned long long ds = f32x2_sub(S[p][k], Cs[k]);
          r2 = k == 0 ? f32x2_mul(df, df) : f32x2_fma(df, df, r2);
          ss = k == 0 ? f32x2_mul(S[p][k], Cs[k]) : f32x2_fma(S[p][k], Cs[k], ss);
          a = f32x2_fma(ds, df, k == 0 ? dd : a);
        }
        const unsigned long long r2m3 = GAUSS ? 0ull : f32x2_mul(r2, m3);
#pragma unroll
        for (int b = 0; b < NS; ++b) {
          float t0, t1;
          f32x2_unpack(GAUSS ? f32x2_mul(r2, P.c2[b]) : f32x2_add(r2, P.c2[b]), t0, t1);
          float k0 = GAUSS ? ex2_neg(t0) : rsqrt_mufu(t0);
          float k1 = GAUSS ? ex2_neg(t1) : rsqrt_mufu(t1);
          if (DIAG) {                                  // i == j: left out of the pair sum
            if (rel == 2 * p * kThreads) k0 = 0.f;
            if (rel == (2 * p + 1) * kThreads) k1 = 0.f;
          }
          const unsigned long long K = f32x2_pack(k0, k1);
          unsigned long long inner;
          if (GAUSS) {
            inner = f32x2_fma(a, P.inv2[b], f32x2_fma(r2, P.ninv4[b], ss));
          } else {
            const unsigned long long K2 = f32x2_mul(K, K);
            inner = f32x2_fma(K2, f32x2_fma(r2m3, K2, a), ss);
          }
          A[p][b] = f32x2_fma(K, inner, A[p][b]);
        }
      }
    };
    int c = 0;
    for (; c + kUnroll <= cnt; c += kUnroll) {
#pragma unroll
      for (int u = 0; u < kUnroll; ++u) column(c + u);
    }
    for (; c < cnt; ++c) column(c);
  }
#pragma unroll
  for (int p = 0; p < NP; ++p)
#pragma unroll
    for (int b = 0; b < NS; ++b) {
      float lo, hi;
      f32x2_unpack(A[p][b], lo, hi);
      if (valid[2 * p]) accd[b] += w * static_cast<double>(lo);
      if (valid[2 * p + 1]) accd[b] += w * static_cast<double>(hi);
    }
}

template <bool GAUSS, int DP, int NS, int RPT>
__global__ void __launch_bounds__(kThreads, ctas_per_sm(DP, NS)) k_ksd(const __grid_constant__ KsdParams P) {
  __shared__ unsigned long long cs[chunk_cols(DP)][2 * DP];
  __shared__ double red[kThreads / 32][2 * NS];
  const long long u_begin = static_cast<long long>(blockIdx.x) * P.u_total / gridDim.x;
  const long long u_end = static_cast<long long>(blockIdx.x + 1) * P.u_total / gridDim.x;
  double accd[2 * NS];
#pragma unroll
  for (int b = 0; b < 2 * NS; ++b) accd[b] = 0.0;
  long long group = -1;
  for (long long u = u_begin; u < u_end; ++u) {
    const long long o = u / P.u_obs;
    long long I, J;
    tri_decode(u - o * P.u_obs, P.t, I, J);
    if (o != group) {
      if (group >= 0) flush_group<2 * NS, kThreads>(accd, P.partial + (blockIdx.x + group) * 2 * NS, red);
      group = o;
    }
    const float* xo = P.x + o * P.n * P.dim;
    const float* so = P.s + o * P.n * P.dim;
    if (I == J)
      tile<GAUSS, DP, NS, RPT, true>(P, xo, so, I, J, 1.0, accd, cs);
    else
      tile<GAUSS, DP, NS, RPT, false>(P, xo, so, I, J, 2.0, accd, cs);
  }
  if (group >= 0) flush_group<2 * NS, kThreads>(accd, P.partial + (blockIdx.x + group) * 2 * NS, red);
}

// One thread per (observation, scale): the off-diagonal and diagonal sums over the CTAs that worked on the observation,
// in CTA order, normalised to {KSD^2_U, KSD^2_V}.
__global__ void k_ksd_finish(const double* __restrict__ partial, long long u_total, long long u_obs, int grid, int n_obs,
                             int ns, long long n, double* out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_obs * ns) return;
  const int o = idx / ns, b = idx - o * ns;
  const long long gb = o * u_obs, ge = gb + u_obs;
  const double off = pairs::sum_group_slots(partial, u_total, grid, o, gb, ge, 2 * ns, b);
  const double dg = pairs::sum_group_slots(partial, u_total, grid, o, gb, ge, 2 * ns, ns + b);
  const double nd = static_cast<double>(n);
  out[2LL * idx] = off / (nd * (nd - 1.0));
  out[2LL * idx + 1] = (off + dg) / (nd * nd);
}

template <bool GAUSS, int DP, int NS>
int run(const KsdParams& P, cudaStream_t s, int* grid_out) {
  auto kern = k_ksd<GAUSS, DP, NS, rows_per_thread(DP, NS)>;
  int dev = 0, sms = 0, occ = 0;
  DMIP_CHECK_CUDA(cudaGetDevice(&dev));
  DMIP_CHECK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  DMIP_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kThreads, 0));
  long long grid = static_cast<long long>(sms) * (occ > 0 ? occ : 1);
  if (grid > kMaxGrid) grid = kMaxGrid;
  if (grid > P.u_total) grid = P.u_total;
  kern<<<static_cast<unsigned>(grid), kThreads, 0, s>>>(P);
  DMIP_CHECK_CUDA(cudaGetLastError());
  *grid_out = static_cast<int>(grid);
  return DMIP_OK;
}

template <bool GAUSS, int DP>
int run_dp(const KsdParams& P, int ns, cudaStream_t s, int* grid) {
  switch (ns) {
    case 1: return run<GAUSS, DP, 1>(P, s, grid);
    case 2: return run<GAUSS, DP, 2>(P, s, grid);
    case 3: return run<GAUSS, DP, 3>(P, s, grid);
    case 4: return run<GAUSS, DP, 4>(P, s, grid);
    case 5: return run<GAUSS, DP, 5>(P, s, grid);
    case 6: return run<GAUSS, DP, 6>(P, s, grid);
    case 7: return run<GAUSS, DP, 7>(P, s, grid);
    default: return run<GAUSS, DP, 8>(P, s, grid);
  }
}

template <bool GAUSS>
int run_kind(const KsdParams& P, int dp, int ns, cudaStream_t s, int* grid) {
  switch (dp) {
    case 1: return run_dp<GAUSS, 1>(P, ns, s, grid);
    case 2: return run_dp<GAUSS, 2>(P, ns, s, grid);
    case 3: return run_dp<GAUSS, 3>(P, ns, s, grid);
    case 4: return run_dp<GAUSS, 4>(P, ns, s, grid);
    case 8: return run_dp<GAUSS, 8>(P, ns, s, grid);
    default: return run_dp<GAUSS, 16>(P, ns, s, grid);
  }
}

}  // namespace

size_t ksd_workspace(const DmipKsd* d) {
  if (!d || d->n_obs < 1 || d->n_scales < 1 || d->n_scales > DMIP_MMD_MAX_BW) return 0;
  return (static_cast<size_t>(kMaxGrid) + static_cast<size_t>(d->n_obs)) * 2 * static_cast<size_t>(d->n_scales) *
         sizeof(double);
}

int launch_ksd(const DmipKsd* d, cudaStream_t s) {
  DMIP_REQUIRE(d->dim >= 1 && d->dim <= DMIP_MMD_MAX_DIM, "KSD dimension must be 1..%d (got %d)", DMIP_MMD_MAX_DIM, d->dim);
  DMIP_REQUIRE(d->n_obs >= 1, "KSD needs n_obs >= 1 (got %d)", d->n_obs);
  DMIP_REQUIRE(d->n >= 2, "KSD needs at least 2 samples per observation (n = %lld)", static_cast<long long>(d->n));
  DMIP_REQUIRE(d->kernel == DMIP_KSD_IMQ || d->kernel == DMIP_KSD_GAUSS,
               "KSD kernel must be DMIP_KSD_IMQ (0) or DMIP_KSD_GAUSS (1) (got %d)", d->kernel);
  DMIP_REQUIRE(d->n_scales >= 1 && d->n_scales <= DMIP_MMD_MAX_BW, "KSD needs 1..%d scales (got %d)", DMIP_MMD_MAX_BW,
               d->n_scales);
  for (int b = 0; b < d->n_scales; ++b)
    DMIP_REQUIRE(d->scale[b] > 0.f && isfinite(d->scale[b]), "scale %d must be positive and finite (got %g)", b,
                 static_cast<double>(d->scale[b]));
  DMIP_REQUIRE(d->x && d->score && d->out, "x / score / out is NULL");
  if (!d->workspace || d->workspace_bytes < ksd_workspace(d)) {
    set_error("workspace too small: need %zu bytes", ksd_workspace(d));
    return DMIP_EWORKSPACE;
  }
  DMIP_REQUIRE((reinterpret_cast<uintptr_t>(d->workspace) & 7) == 0, "workspace must be 8-byte aligned");

  const bool gauss = d->kernel == DMIP_KSD_GAUSS;
  auto dup = [](double v) {   // (v, v) as a packed fp32 pair
    const float f = static_cast<float>(v);
    uint32_t u;
    memcpy(&u, &f, 4);
    return (static_cast<unsigned long long>(u) << 32) | u;
  };
  KsdParams P = {};
  P.x = d->x;
  P.s = d->score;
  P.n = d->n;
  P.dim = d->dim;
  for (int b = 0; b < d->n_scales; ++b) {
    const double c = d->scale[b], c2 = c * c;
    if (gauss) {
      P.c2[b] = dup(1.4426950408889634 / (2.0 * c2));
      P.inv2[b] = dup(1.0 / c2);
      P.ninv4[b] = dup(-1.0 / (c2 * c2));
      P.diag_a[b] = 1.0;
      P.diag_b[b] = d->dim / c2;
    } else {
      P.c2[b] = dup(c2);
      P.diag_a[b] = 1.0 / c;
      P.diag_b[b] = d->dim / (c2 * c);
    }
  }
  const int dp = d->dim <= 4 ? d->dim : d->dim <= 8 ? 8 : 16;
  const long long T = kThreads * rows_per_thread(dp, d->n_scales);
  P.t = (d->n + T - 1) / T;
  P.u_obs = P.t * (P.t + 1) / 2;
  P.u_total = P.u_obs * d->n_obs;
  P.partial = static_cast<double*>(d->workspace);

  int grid = 0;
  const int rc = gauss ? run_kind<true>(P, dp, d->n_scales, s, &grid) : run_kind<false>(P, dp, d->n_scales, s, &grid);
  if (rc) return rc;
  count_launch();
  const int nthreads = d->n_obs * d->n_scales;
  k_ksd_finish<<<(nthreads + 127) / 128, 128, 0, s>>>(P.partial, P.u_total, P.u_obs, grid, d->n_obs, d->n_scales, d->n,
                                                      d->out);
  DMIP_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return DMIP_OK;
}

}  // namespace dmip
