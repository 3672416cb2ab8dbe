// dmip_surrogate.cu — K4: forward + reverse sweep through the frozen scatterometry surrogate (ReLU MLP
// 3 -> 256 -> 256 -> 256 -> 23, utils_scatterometry.py:9-16) fused with the cotangent that feeds it.
//
//   mode 0  energy E(x) = 1/2 sum log p + 1/2 sum (y-f)^2/p + lambd_bd sum [relu(x-1) + relu(-1-x)],
//           p = (a f)^2 + b^2  (get_log_posterior, utils_scatterometry.py:30-38) and grad_x E
//           (energy_grad, models/SNF.py:234-237); score_posterior = -grad_x E is the PINNLoss initial condition
//           (main_diffusion_scatterometry.py:142-145).  Closed form: SURVEY.md App. A.6.
//   mode 1  u = J_f(x)^T w with w = -a^2 f/p + (y-f)/p + a^2 (y-f)^2 f/p — the three VJPs of
//           PosteriorLoss.likelihood_target (losses.py:349-371) merged into one sweep.
//
// One CTA = 32 rows.  The ReLU masks of the hidden layers are kept as one 32-bit word per (layer, unit) in shared
// memory; the reverse sweep reuses the untransposed nn.Linear weights as [contraction][output].
#include "dmip_common.h"
#include "dmip_tile.cuh"
#include "dmip_rng.cuh"

namespace dmip {

namespace {

struct SurrDev {
  int mode, n_layers, in_dim, out_dim;
  int width[DMIP_MAX_LAYERS];
  const float* W[DMIP_MAX_LAYERS];
  const float* Wt[DMIP_MAX_LAYERS];
  const float* b[DMIP_MAX_LAYERS];
  float a, bb, lambd;
  long long n;
  long long rpo;        // rows per observation (0: one y row per x row)
  const float* x;
  const float* y;
  float* energy;
  float* grad;
  float* fx;
};

__global__ void __launch_bounds__(kThreadsL, 1) k_surrogate(const __grid_constant__ SurrDev P) {
  extern __shared__ __align__(16) float smem[];
  float* buf0 = smem;
  float* buf1 = smem + kMaxW * kLd;
  float* wbuf = buf1 + kMaxW * kLd;                                     // weight slabs of the staged GEMM
  uint32_t* masks = reinterpret_cast<uint32_t*>(wbuf + kWbufFloats);    // [n_layers-1][kMaxW]
  const int t = threadIdx.x, lane = t & 31;
  const long long n_tiles = (P.n + kRows - 1) / kRows;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long r0 = tile * kRows;
    for (int idx = t; idx < kRows * P.in_dim; idx += kThreadsL) {
      const int k = idx / kRows, r = idx % kRows;
      buf0[k * kLd + r] = (r0 + r < P.n) ? P.x[(r0 + r) * P.in_dim + k] : 0.f;
    }
    __syncthreads();
    float* in = buf0;
    float* out = buf1;
    int K = P.in_dim;
    const int L = P.n_layers - 1;
    for (int l = 0; l <= L; ++l) {
      const int N = P.width[l];
      tile_gemm(in, out, P.Wt[l], K, N, wbuf);
      for (int idx = t; idx < N * kRows; idx += kThreadsL) {      // a warp = one unit n, lane = row
        const int n = idx >> 5;
        float z = out[n * kLd + lane] + P.b[l][n];
        if (l < L) {
          const uint32_t m = __ballot_sync(0xffffffffu, z > 0.f);
          if (lane == 0) masks[l * kMaxW + n] = m;
          z = fmaxf(z, 0.f);
        }
        out[n * kLd + lane] = z;
      }
      __syncthreads();
      float* tmp = in; in = out; out = tmp;
      K = N;
    }
    // ---- per-row energy and cotangent d(.)/df  (in: f[j][row])
    if (t < kRows) {
      const long long row = r0 + t;
      const bool live = row < P.n;
      const float a2 = P.a * P.a;
      float E = 0.f;
      for (int j = 0; j < P.out_dim; ++j) {
        const float f = in[j * kLd + t];
        const float yv = live ? P.y[(P.rpo > 0 ? row / P.rpo : row) * P.out_dim + j] : 0.f;
        const float p = a2 * f * f + P.bb * P.bb;
        const float r = yv - f;
        float w;
        if (P.mode == 0) {
          E += 0.5f * logf(p) + 0.5f * r * r / p;
          w = a2 * f / p - r / p - a2 * f * r * r / (p * p);       // dE/df  (App. A.6)
        } else {
          w = -a2 * f / p + r / p + a2 * r * r * f / p;            // -a^2 v1 + v2 + a^2 v3  (losses.py:354-368)
        }
        if (live && P.fx) P.fx[row * P.out_dim + j] = f;
        in[j * kLd + t] = w;
      }
      if (P.mode == 0 && live && P.energy) {
        for (int k = 0; k < P.in_dim; ++k) {
          const float xv = P.x[row * P.in_dim + k];
          E += P.lambd * (fmaxf(xv - 1.f, 0.f) + fmaxf(-1.f - xv, 0.f));
        }
        P.energy[row] = E;
      }
    }
    __syncthreads();
    // ---- reverse sweep
    for (int l = L; l >= 0; --l) {
      const int N = P.width[l];
      const int Kp = (l == 0) ? P.in_dim : P.width[l - 1];
      tile_gemm(in, out, P.W[l], N, Kp, wbuf);
      if (l > 0) {
        for (int idx = t; idx < Kp * kRows; idx += kThreadsL) {
          const int k = idx >> 5;
          if (!((masks[(l - 1) * kMaxW + k] >> lane) & 1u)) out[k * kLd + lane] = 0.f;
        }
        __syncthreads();
      }
      float* tmp = in; in = out; out = tmp;
    }
    for (int idx = t; idx < kRows * P.in_dim; idx += kThreadsL) {
      const int r = idx / P.in_dim, k = idx % P.in_dim;
      const long long row = r0 + r;
      if (row < P.n) {
        float g = in[k * kLd + r];
        if (P.mode == 0) {
          const float xv = P.x[row * P.in_dim + k];
          g += P.lambd * ((xv > 1.f ? 1.f : 0.f) - (xv < -1.f ? 1.f : 0.f));
        }
        P.grad[row * P.in_dim + k] = g;
      }
    }
    __syncthreads();
  }
}


// ------------------------------------------------------------------------------------------------ Metropolis chains
// anneal_to_energy (models/SNF.py:250-275, langevin_prop=False) as it is used to produce the scatterometry ground-truth
// samples (generate_scatterometry_ground_truth.py:26-29): random-walk Metropolis on E(x) = get_log_posterior.  One CTA =
// 32 chains for ALL steps: the chain state and its energy stay in registers of the chain's thread, each step is one
// surrogate forward of the proposals (the reference evaluates E(x_curr) again every step; it is cached here).
constexpr int kStreamMcmcNoise = 2;   // Philox stream ids (0/1 are the sampler's, dmip_rng.cuh)
constexpr int kStreamMcmcUnif = 3;
constexpr int kMaxChainDim = 8;

struct MetroDev {
  SurrDev S;                 // net, a, b, lambd, n (= chains), y (n_obs, out_dim)
  long long n_per_obs;
  int steps;
  float noise_std;
  float* xio;                // (n, in_dim) start points in, final points out
  float* de;                 // (n,) E(final) - E(start) or NULL
  int rng_mode;
  unsigned long long seed, gidx_base;
  const float* noise;        // injected: (steps, n, in_dim)
  const float* unif;         // injected: (steps, n)
};

__global__ void __launch_bounds__(kThreadsL, 1) k_metropolis(const __grid_constant__ MetroDev M) {
  extern __shared__ __align__(16) float smem[];
  float* buf0 = smem;
  float* buf1 = smem + kMaxW * kLd;
  float* wbuf = buf1 + kMaxW * kLd;
  const SurrDev& P = M.S;
  const int t = threadIdx.x, lane = t & 31;
  const int dim = P.in_dim, L = P.n_layers - 1;
  const long long n_tiles = (P.n + kRows - 1) / kRows;
  const float a2 = P.a * P.a, b2 = P.bb * P.bb;

  // forward through the surrogate for the 32 points in buf0; returns the buffer holding f[j][row]
  auto forward = [&]() -> float* {
    float* in = buf0;
    float* out = buf1;
    int K = dim;
    for (int l = 0; l <= L; ++l) {
      const int N = P.width[l];
      tile_gemm(in, out, P.Wt[l], K, N, wbuf);
      for (int idx = t; idx < N * kRows; idx += kThreadsL) {
        const int n = idx >> 5;
        const float z = out[n * kLd + lane] + P.b[l][n];
        out[n * kLd + lane] = (l < L) ? fmaxf(z, 0.f) : z;
      }
      __syncthreads();
      float* tmp = in; in = out; out = tmp;
      K = N;
    }
    return in;
  };
  // get_log_posterior of the chain's point xe from f = fb[.][t]      (utils_scatterometry.py:30-38)
  auto energy = [&](const float* fb, const float* yrow, const float (&xe)[kMaxChainDim]) {
    float E = 0.f;
    for (int j = 0; j < P.out_dim; ++j) {
      const float f = fb[j * kLd + t];
      const float p = a2 * f * f + b2;
      const float r = yrow[j] - f;
      E += 0.5f * logf(p) + 0.5f * r * r / p;
    }
#pragma unroll
    for (int k = 0; k < kMaxChainDim; ++k)
      if (k < dim) E += P.lambd * (fmaxf(xe[k] - 1.f, 0.f) + fmaxf(-1.f - xe[k], 0.f));
    return E;
  };

  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long row = tile * kRows + t;
    const bool owner = t < kRows, live = owner && row < P.n;
    const float* yrow = P.y + (live ? row / M.n_per_obs : 0) * P.out_dim;
    float xc[kMaxChainDim], xp[kMaxChainDim];
    float e_cur = 0.f, e0 = 0.f;
    if (owner) {
#pragma unroll
      for (int k = 0; k < kMaxChainDim; ++k)
        if (k < dim) {
          xc[k] = live ? M.xio[row * dim + k] : 0.f;
          buf0[k * kLd + t] = xc[k];
        }
    }
    __syncthreads();
    {
      const float* fb = forward();
      if (owner) e0 = e_cur = energy(fb, yrow, xc);
    }
    for (int step = 0; step < M.steps; ++step) {
      float u = 1.f;
      if (owner) {
        float z[kMaxChainDim];
        if (M.rng_mode == DMIP_RNG_INJECTED) {
#pragma unroll
          for (int k = 0; k < kMaxChainDim; ++k)
            if (k < dim) z[k] = live ? M.noise[(static_cast<long long>(step) * P.n + row) * dim + k] : 0.f;
          u = live ? M.unif[static_cast<long long>(step) * P.n + row] : 1.f;
        } else {
          const unsigned long long gidx = M.gidx_base + static_cast<unsigned long long>(row);
#pragma unroll
          for (int q = 0; q < kMaxChainDim / 4; ++q)
            if (4 * q < dim) {
              float zz[4];
              philox_normal4(gidx, static_cast<uint32_t>(step), kStreamMcmcNoise, q, M.seed, zz);
#pragma unroll
              for (int e = 0; e < 4; ++e) z[4 * q + e] = zz[e];
            }
          uint32_t r[4];
          philox4x32_10(static_cast<uint32_t>(gidx), static_cast<uint32_t>(gidx >> 32), static_cast<uint32_t>(step),
                        static_cast<uint32_t>(kStreamMcmcUnif) << 16, static_cast<uint32_t>(M.seed),
                        static_cast<uint32_t>(M.seed >> 32), r);
          u = u01(r[0]);
        }
#pragma unroll
        for (int k = 0; k < kMaxChainDim; ++k)
          if (k < dim) {
            xp[k] = xc[k] + M.noise_std * z[k];                       // SNF.py:259-260
            buf0[k * kLd + t] = xp[k];
          }
      }
      __syncthreads();
      const float* fb = forward();
      if (owner) {
        const float e_prop = energy(fb, yrow, xp);
        if (u < expf(-e_prop + e_cur)) {                              // acc = r < exp(-e_prop + e_curr)   (:264-268)
          e_cur = e_prop;
#pragma unroll
          for (int k = 0; k < kMaxChainDim; ++k)
            if (k < dim) xc[k] = xp[k];
        }
      }
      // the owner threads rewrite only their own column of buf0 next; everyone meets again at the barrier above
    }
    if (live) {
#pragma unroll
      for (int k = 0; k < kMaxChainDim; ++k)
        if (k < dim) M.xio[row * dim + k] = xc[k];
      if (M.de) M.de[row] = e_cur - e0;
    }
    __syncthreads();
  }
}

// the net part of the device descriptor: transposed weights in the workspace, the untransposed ones for the reverse sweep
int stage_surrogate_net(const DmipMlp& net, void* ws, SurrDev* P, cudaStream_t s) {
  for (int l = 0; l < net.n_layers; ++l) P->W[l] = net.W[l];
  return tile_net_stage(net, ws, P, s);
}

}  // namespace

size_t metropolis_workspace(const DmipMetropolis* d) { return tile_net_bytes(d->net); }

int launch_metropolis(const DmipMetropolis* d, cudaStream_t s) {
  int rc = tile_net_check(d->net, d->net.in_dim, "surrogate");
  if (rc) return rc;
  DMIP_REQUIRE(d->net.in_dim <= kMaxChainDim, "Metropolis chains: state dimension must be <= %d", kMaxChainDim);
  DMIP_REQUIRE(d->n_obs >= 0 && d->n_per_obs >= 0 && d->steps >= 0, "n_obs / n_per_obs / steps must be >= 0");
  DMIP_REQUIRE(d->rng_mode == DMIP_RNG_PHILOX || d->rng_mode == DMIP_RNG_INJECTED, "rng_mode must be philox or injected");
  const long long n = static_cast<long long>(d->n_obs) * d->n_per_obs;
  if (n == 0) return DMIP_OK;
  DMIP_REQUIRE(d->x && d->y, "x / y is NULL");
  DMIP_REQUIRE(d->rng_mode != DMIP_RNG_INJECTED || d->steps == 0 || (d->noise && d->unif),
               "injected rng_mode needs noise (steps, n, xdim) and unif (steps, n)");
  if (!d->workspace || d->workspace_bytes < metropolis_workspace(d)) {
    set_error("workspace too small: need %zu bytes", metropolis_workspace(d));
    return DMIP_EWORKSPACE;
  }
  static int n_sm = 0;
  static bool ready[64] = {};
  const int smem = (2 * kMaxW * kLd + kWbufFloats) * 4;
  int dev = 0;
  DMIP_CHECK_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || !ready[dev]) {
    DMIP_CHECK_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
    DMIP_CHECK_CUDA(cudaFuncSetAttribute(k_metropolis, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    if (dev >= 0 && dev < 64) ready[dev] = true;
  }
  MetroDev M = {};
  if ((rc = stage_surrogate_net(d->net, d->workspace, &M.S, s))) return rc;
  M.S.a = d->a; M.S.bb = d->b; M.S.lambd = d->lambd_bd;
  M.S.n = n;
  M.S.y = d->y;
  M.n_per_obs = d->n_per_obs;
  M.steps = d->steps;
  M.noise_std = d->noise_std;
  M.xio = d->x;
  M.de = d->de;
  M.rng_mode = d->rng_mode;
  M.seed = d->seed;
  M.gidx_base = d->gidx_base;
  M.noise = d->noise;
  M.unif = d->unif;
  const long long tiles = (n + kRows - 1) / kRows;
  k_metropolis<<<static_cast<unsigned>(tiles), kThreadsL, smem, s>>>(M);
  DMIP_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return DMIP_OK;
}

// [transposed fp32 weights of the FFMA kernel | packed bf16 hi / lo images of the tensor-core kernel], each part 1 KB aligned
static size_t surrogate_ffma_bytes(const DmipSurrogate* d) {
  return (tile_net_bytes(d->net) + 1023) / 1024 * 1024;
}
size_t surrogate_workspace(const DmipSurrogate* d) { return surrogate_ffma_bytes(d) + surrogate_tc_workspace() + 1024; }

int launch_surrogate(const DmipSurrogate* d, cudaStream_t s) {
  const DmipMlp& net = d->net;
  int rc = tile_net_check(net, net.in_dim, "surrogate");
  if (rc) return rc;
  DMIP_REQUIRE(d->mode == 0 || d->mode == 1, "surrogate mode must be 0 (energy + gradient) or 1 (likelihood VJP)");
  DMIP_REQUIRE(d->n >= 0 && d->rows_per_obs >= 0, "negative row count / rows_per_obs");
  if (d->n == 0) return DMIP_OK;
  DMIP_REQUIRE(d->x && d->y && d->grad, "x / y / grad is NULL");
  if (!d->workspace || d->workspace_bytes < surrogate_workspace(d)) {
    set_error("workspace too small: need %zu bytes", surrogate_workspace(d));
    return DMIP_EWORKSPACE;
  }
  if (surrogate_tc_supported(net)) {
    // tcgen05 path (dmip_surrogate_tc.cu): its weight images sit behind the FFMA kernel's part, at the next 1 KB boundary
    const uintptr_t base = reinterpret_cast<uintptr_t>(d->workspace) + surrogate_ffma_bytes(d);
    return launch_surrogate_tc(d, reinterpret_cast<void*>((base + 1023) / 1024 * 1024), s);
  }
  static int n_sm = 0;
  static bool ready[64] = {};   // cudaFuncSetAttribute is per device
  const int smem = (2 * kMaxW * kLd + kWbufFloats) * 4 + (DMIP_MAX_LAYERS - 1) * kMaxW * 4;
  int dev = 0;
  DMIP_CHECK_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || !ready[dev]) {
    DMIP_CHECK_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
    DMIP_CHECK_CUDA(cudaFuncSetAttribute(k_surrogate, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    if (dev >= 0 && dev < 64) ready[dev] = true;
  }
  SurrDev P = {};
  P.mode = d->mode;
  if ((rc = stage_surrogate_net(net, d->workspace, &P, s))) return rc;
  P.a = d->a;
  P.bb = d->b;
  P.lambd = d->lambd_bd;
  P.n = d->n;
  P.rpo = d->rows_per_obs;
  P.x = d->x;
  P.y = d->y;
  P.energy = d->energy;
  P.grad = d->grad;
  P.fx = d->fx;
  const long long tiles = (d->n + kRows - 1) / kRows;
  k_surrogate<<<static_cast<unsigned>(tiles < 4LL * n_sm ? tiles : 4LL * n_sm), kThreadsL, smem, s>>>(P);
  DMIP_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return DMIP_OK;
}

}  // namespace dmip
