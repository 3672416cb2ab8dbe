// dmip_mmd.cu — unbiased Gaussian-kernel MMD^2 between two sample sets per observation (Gretton et al. 2012, JMLR 13,
// eq. 3), for up to DMIP_MMD_MAX_BW bandwidths at once.  No reference counterpart: the reference reports only the
// histogram KL (dmip_metrics.cu).
//
// For k_b(a, c) = exp(-|a - c|^2 / (2 sigma_b^2)) = 2^(-s^2 |a - c|^2 r_b) with s^2 = log2(e) / (2 sigma_0^2) and
// r_b = sigma_0^2 / sigma_b^2, every point is scaled by s once on load; a pair then costs d packed FADD2 + d packed FFMA2
// per two rows, and per bandwidth one FMUL2 (b > 0), one MUFU.EX2 per pair and one FADD2 per two pairs.  The MUFU
// (16 lanes/clk/SM) is the roofline; the FP32 side stays below it (DESIGN.md §3 "Evaluation metrics", which also records
// why a polynomial exp2 on the FMA pipe for part of the pairs was measured and not kept).
//
// Work: per observation the XX and YY terms visit the tiles I <= J of their square (T x T) tiling, the XY term every
// tile.  A work unit is one (observation, term, I, J) tile; the units are numbered observation-major and every CTA of the
// persistent grid takes one contiguous range of them (static, so the summation order is fixed and results are
// bit-identical from run to run on one device).  Each thread holds RPT rows in registers and streams the tile's columns
// through shared memory in chunks of 256; per-row fp32 sums cover at most T columns and are folded into per-thread fp64
// sums after every unit (x2 for off-diagonal XX / YY tiles, whose mirror tile is not visited).  When the CTA leaves a
// (observation, term) group it reduces those fp64 sums over the block in a fixed order into workspace slot
// [cta + group]: the (cta, group) pairs a contiguous partition produces are a staircase, so cta + group is unique.
// k_mmd_finish sums the slots of each group in CTA order and normalises.  Two launches per call.
#include <float.h>
#include <math.h>

#include "dmip_common.h"
#include "dmip_ptx.cuh"

namespace dmip {

namespace {

constexpr int kThreads = 256;
constexpr int kChunk = kThreads;   // columns staged in shared memory at a time (one per thread)
constexpr int kUnroll = 4;         // column loop unroll; chunks are padded to a multiple with far-away sentinels
constexpr int kMaxGrid = 1024;     // bounds the workspace independently of the device
constexpr float kFar = 1e30f;      // sentinel coordinate: the squared distance overflows to +inf and the kernel value is 0

// rows held per thread (the tile edge is 256 x this): as many as fit 128 registers without spilling (two CTAs per SM)
constexpr int rows_per_thread(int dp, int nb) {
  return dp <= 4 ? (nb <= 5 ? 8 : dp * nb <= 28 ? 4 : 2) : dp == 8 ? (nb <= 5 ? 4 : 2) : 2;
}

struct MmdParams {
  const float* x;                 // (n_obs, n, dim)
  const float* y;                 // (n_obs, m, dim)
  long long n, m;
  int dim;
  float scale;                    // s = sqrt(log2(e) / (2 sigma_0^2))
  float ratio[DMIP_MMD_MAX_BW];   // r_b = sigma_0^2 / sigma_b^2
  long long tx, ty;               // tiles along x / y
  long long u_xx, u_yy, u_obs;    // units of the XX and YY terms and of one observation (XY = u_obs - u_xx - u_yy)
  long long u_total;
  double* partial;                // (kMaxGrid + 3 n_obs) x n_bw fp64 slots
};

__device__ __forceinline__ float ex2_neg(float t) {   // 2^-t on the MUFU
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(-t));
  return r;
}
// row index I and column index J >= I of unit r of the upper triangle (row-major) of a t x t tiling
__device__ __forceinline__ void tri_decode(long long r, long long t, long long& I, long long& J) {
  const double b = 2.0 * static_cast<double>(t) + 1.0;
  long long i = static_cast<long long>((b - sqrt(b * b - 8.0 * static_cast<double>(r))) * 0.5);
  auto off = [t](long long k) { return k * t - k * (k - 1) / 2; };
  if (i < 0) i = 0;
  if (i > t - 1) i = t - 1;
  while (i > 0 && off(i) > r) --i;
  while (i + 1 < t && off(i + 1) <= r) ++i;
  I = i;
  J = i + (r - off(i));
}

template <int NB>
__device__ __forceinline__ void flush_group(double (&acc)[NB], double* slot, double (*red)[NB]) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int b = 0; b < NB; ++b) {
    double v = acc[b];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[warp][b] = v;
    acc[b] = 0.0;
  }
  __syncthreads();
  if (threadIdx.x < NB) {
    double s = 0.0;
    for (int w = 0; w < kThreads / 32; ++w) s += red[w][threadIdx.x];
    slot[threadIdx.x] = s;
  }
  __syncthreads();
}

// One T x T tile: rows [I T, I T + T) of `rows` against columns [J T, J T + T) of `cols`.
template <int DP, int NB, int RPT, bool DIAG>
__device__ __forceinline__ void tile(const MmdParams& P, const float* __restrict__ rows, long long nr,
                                     const float* __restrict__ cols, long long nc, long long I, long long J, double w,
                                     double (&accd)[NB], unsigned long long (*cs)[DP]) {
  constexpr int T = kThreads * RPT, NP = RPT / 2;
  const int tid = threadIdx.x;
  const int dim = P.dim;
  const float s = P.scale;
  unsigned long long R[NP][DP];
  bool valid[RPT];
#pragma unroll
  for (int p = 0; p < NP; ++p) {
    float v[2][DP];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const long long i = I * T + static_cast<long long>(2 * p + h) * kThreads + tid;
      valid[2 * p + h] = i < nr;
#pragma unroll
      for (int k = 0; k < DP; ++k)
        v[h][k] = (i < nr && (DP <= 4 || k < dim)) ? __ldg(rows + i * dim + k) * s : 0.f;
    }
#pragma unroll
    for (int k = 0; k < DP; ++k) R[p][k] = f32x2_pack(v[0][k], v[1][k]);
  }
  unsigned long long rb[NB];
#pragma unroll
  for (int b = 0; b < NB; ++b) rb[b] = f32x2_pack(P.ratio[b], P.ratio[b]);
  unsigned long long A[NP][NB];
#pragma unroll
  for (int p = 0; p < NP; ++p)
#pragma unroll
    for (int b = 0; b < NB; ++b) A[p][b] = 0ull;

  const long long c0 = J * T;
  const int ncol = static_cast<int>(nc - c0 < T ? nc - c0 : T);
  for (int ch = 0; ch < ncol; ch += kChunk) {
    const int cnt = ncol - ch < kChunk ? ncol - ch : kChunk;
    const int cntp = (cnt + kUnroll - 1) / kUnroll * kUnroll;
    __syncthreads();                                   // the previous chunk's readers are done
    if (tid < cntp) {
      const long long j = c0 + ch + tid;
#pragma unroll
      for (int k = 0; k < DP; ++k) {
        const float v = tid < cnt ? ((DP <= 4 || k < dim) ? -__ldg(cols + j * dim + k) * s : 0.f) : kFar;
        cs[tid][k] = f32x2_pack(v, v);
      }
    }
    __syncthreads();
    const int qd = ch / kChunk;                        // DIAG: the row slot whose rows are this chunk's columns
    for (int c = 0; c < cntp; c += kUnroll) {
#pragma unroll
      for (int u = 0; u < kUnroll; ++u) {
        unsigned long long C[DP];
#pragma unroll
        for (int k = 0; k < DP; ++k) C[k] = cs[c + u][k];
#pragma unroll
        for (int p = 0; p < NP; ++p) {
          unsigned long long dist = 0ull;
#pragma unroll
          for (int k = 0; k < DP; ++k) {
            const unsigned long long df = f32x2_add(R[p][k], C[k]);
            dist = k == 0 ? f32x2_mul(df, df) : f32x2_fma(df, df, dist);
          }
          if (DIAG && c + u == tid) {                  // i == j: excluded from the XX / YY means
            if (qd == 2 * p) dist = (dist & 0xffffffff00000000ull) | 0x7f800000ull;
            if (qd == 2 * p + 1) dist = (dist & 0x00000000ffffffffull) | (0x7f800000ull << 32);
          }
#pragma unroll
          for (int b = 0; b < NB; ++b) {
            const unsigned long long t = b == 0 ? dist : f32x2_mul(dist, rb[b]);
            float t0, t1;
            f32x2_unpack(t, t0, t1);
            A[p][b] = f32x2_add(A[p][b], f32x2_pack(ex2_neg(t0), ex2_neg(t1)));
          }
        }
      }
    }
  }
#pragma unroll
  for (int p = 0; p < NP; ++p)
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      float lo, hi;
      f32x2_unpack(A[p][b], lo, hi);
      if (valid[2 * p]) accd[b] += w * static_cast<double>(lo);
      if (valid[2 * p + 1]) accd[b] += w * static_cast<double>(hi);
    }
}

template <int DP, int NB, int RPT>
__global__ void __launch_bounds__(kThreads, 2) k_mmd(const __grid_constant__ MmdParams P) {
  __shared__ unsigned long long cs[kChunk][DP];
  __shared__ double red[kThreads / 32][NB];
  const long long u_begin = static_cast<long long>(blockIdx.x) * P.u_total / gridDim.x;
  const long long u_end = static_cast<long long>(blockIdx.x + 1) * P.u_total / gridDim.x;
  double accd[NB];
#pragma unroll
  for (int b = 0; b < NB; ++b) accd[b] = 0.0;
  long long group = -1;
  for (long long u = u_begin; u < u_end; ++u) {
    const long long o = u / P.u_obs;
    long long r = u - o * P.u_obs, I, J;
    int term;
    if (r < P.u_xx) {
      term = 0;
      tri_decode(r, P.tx, I, J);
    } else if ((r -= P.u_xx) < P.u_yy) {
      term = 1;
      tri_decode(r, P.ty, I, J);
    } else {
      r -= P.u_yy;
      term = 2;
      I = r / P.ty;
      J = r - I * P.ty;
    }
    const long long g = 3 * o + term;
    if (g != group) {
      if (group >= 0) flush_group<NB>(accd, P.partial + (blockIdx.x + group) * NB, red);
      group = g;
    }
    const float* xo = P.x + o * P.n * P.dim;
    const float* yo = P.y + o * P.m * P.dim;
    const float* rows = term == 1 ? yo : xo;
    const float* cols = term == 0 ? xo : yo;
    const long long nr = term == 1 ? P.m : P.n, nc = term == 0 ? P.n : P.m;
    if (term != 2 && I == J)
      tile<DP, NB, RPT, true>(P, rows, nr, cols, nc, I, J, 1.0, accd, cs);
    else
      tile<DP, NB, RPT, false>(P, rows, nr, cols, nc, I, J, term == 2 ? 1.0 : 2.0, accd, cs);
  }
  if (group >= 0) flush_group<NB>(accd, P.partial + (blockIdx.x + group) * NB, red);
}

// One thread per (observation, bandwidth): the group sums over the CTAs that worked on the group, in CTA order.
__global__ void k_mmd_finish(const double* __restrict__ partial, long long u_total, long long u_obs, long long u_xx,
                             long long u_yy, int grid, int n_obs, int nb, long long n, long long m, double* out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_obs * nb) return;
  const int o = idx / nb, b = idx - o * nb;
  double S[3];
  for (int term = 0; term < 3; ++term) {
    const long long g = 3LL * o + term;
    const long long gb = o * u_obs + (term > 0 ? u_xx : 0) + (term > 1 ? u_yy : 0);
    const long long ge = term == 0 ? gb + u_xx : term == 1 ? gb + u_yy : (o + 1) * u_obs;
    double s = 0.0;
    for (int c = 0; c < grid; ++c) {
      const long long cb = static_cast<long long>(c) * u_total / grid, ce = static_cast<long long>(c + 1) * u_total / grid;
      if (cb < ge && ce > gb) s += partial[(c + g) * nb + b];
    }
    S[term] = s;
  }
  const double kxx = S[0] / (static_cast<double>(n) * static_cast<double>(n - 1));
  const double kyy = S[1] / (static_cast<double>(m) * static_cast<double>(m - 1));
  const double kxy = S[2] / (static_cast<double>(n) * static_cast<double>(m));
  double* q = out + static_cast<long long>(idx) * 4;
  q[0] = kxx + kyy - 2.0 * kxy;
  q[1] = kxx;
  q[2] = kyy;
  q[3] = kxy;
}

template <int DP, int NB>
int run(const MmdParams& P, cudaStream_t s, int* grid_out) {
  auto kern = k_mmd<DP, NB, rows_per_thread(DP, NB)>;
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

template <int DP>
int run_dp(const MmdParams& P, int nb, cudaStream_t s, int* grid) {
  switch (nb) {
    case 1: return run<DP, 1>(P, s, grid);
    case 2: return run<DP, 2>(P, s, grid);
    case 3: return run<DP, 3>(P, s, grid);
    case 4: return run<DP, 4>(P, s, grid);
    case 5: return run<DP, 5>(P, s, grid);
    case 6: return run<DP, 6>(P, s, grid);
    case 7: return run<DP, 7>(P, s, grid);
    default: return run<DP, 8>(P, s, grid);
  }
}

}  // namespace

size_t mmd_workspace(const DmipMmd* d) {
  if (!d || d->n_obs < 1 || d->n_bw < 1 || d->n_bw > DMIP_MMD_MAX_BW) return 0;
  return (static_cast<size_t>(kMaxGrid) + 3 * static_cast<size_t>(d->n_obs)) * static_cast<size_t>(d->n_bw) * sizeof(double);
}

int launch_mmd(const DmipMmd* d, cudaStream_t s) {
  DMIP_REQUIRE(d->dim >= 1 && d->dim <= DMIP_MMD_MAX_DIM, "MMD dimension must be 1..%d (got %d)", DMIP_MMD_MAX_DIM, d->dim);
  DMIP_REQUIRE(d->n_obs >= 1, "MMD needs n_obs >= 1 (got %d)", d->n_obs);
  DMIP_REQUIRE(d->n >= 2 && d->m >= 2, "MMD needs at least 2 samples per set (n = %lld, m = %lld)",
               static_cast<long long>(d->n), static_cast<long long>(d->m));
  DMIP_REQUIRE(d->n_bw >= 1 && d->n_bw <= DMIP_MMD_MAX_BW, "MMD needs 1..%d bandwidths (got %d)", DMIP_MMD_MAX_BW,
               d->n_bw);
  for (int b = 0; b < d->n_bw; ++b)
    DMIP_REQUIRE(d->sigma[b] > 0.f && isfinite(d->sigma[b]), "bandwidth %d must be positive and finite (got %g)", b,
                 static_cast<double>(d->sigma[b]));
  DMIP_REQUIRE(d->x && d->y && d->out, "x / y / out is NULL");
  if (!d->workspace || d->workspace_bytes < mmd_workspace(d)) {
    set_error("workspace too small: need %zu bytes", mmd_workspace(d));
    return DMIP_EWORKSPACE;
  }
  DMIP_REQUIRE((reinterpret_cast<uintptr_t>(d->workspace) & 7) == 0, "workspace must be 8-byte aligned");

  MmdParams P = {};
  P.x = d->x;
  P.y = d->y;
  P.n = d->n;
  P.m = d->m;
  P.dim = d->dim;
  const double s0 = d->sigma[0];
  P.scale = static_cast<float>(sqrt(1.4426950408889634 / (2.0 * s0 * s0)));
  for (int b = 0; b < d->n_bw; ++b) {
    const double r = (s0 / d->sigma[b]) * (s0 / d->sigma[b]);
    P.ratio[b] = static_cast<float>(r < FLT_MAX ? r : FLT_MAX);   // 0 * FLT_MAX = 0 keeps coincident points at k = 1
  }
  const int dp = d->dim <= 4 ? d->dim : d->dim <= 8 ? 8 : 16;
  const long long T = kThreads * rows_per_thread(dp, d->n_bw);
  P.tx = (d->n + T - 1) / T;
  P.ty = (d->m + T - 1) / T;
  P.u_xx = P.tx * (P.tx + 1) / 2;
  P.u_yy = P.ty * (P.ty + 1) / 2;
  P.u_obs = P.u_xx + P.u_yy + P.tx * P.ty;
  P.u_total = P.u_obs * d->n_obs;
  P.partial = static_cast<double*>(d->workspace);

  int grid = 0, rc;
  switch (dp) {
    case 1: rc = run_dp<1>(P, d->n_bw, s, &grid); break;
    case 2: rc = run_dp<2>(P, d->n_bw, s, &grid); break;
    case 3: rc = run_dp<3>(P, d->n_bw, s, &grid); break;
    case 4: rc = run_dp<4>(P, d->n_bw, s, &grid); break;
    case 8: rc = run_dp<8>(P, d->n_bw, s, &grid); break;
    default: rc = run_dp<16>(P, d->n_bw, s, &grid); break;
  }
  if (rc) return rc;
  count_launch();
  const int nthreads = d->n_obs * d->n_bw;
  k_mmd_finish<<<(nthreads + 127) / 128, 128, 0, s>>>(P.partial, P.u_total, P.u_obs, P.u_xx, P.u_yy, grid, d->n_obs,
                                                        d->n_bw, d->n, d->m, d->out);
  DMIP_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return DMIP_OK;
}

}  // namespace dmip
