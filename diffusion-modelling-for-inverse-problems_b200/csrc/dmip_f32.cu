// dmip_f32.cu — the fp32 (FFMA) path: the same fused sampler / forward as dmip_tc.cu for ANY layer widths
// (<= 512) and to fp32 round-off of the reference (accurate tanhf, no operand rounding).  It is the strict-
// parity mode of the product and the GPU-side cross-check of the tcgen05 path at sizes the CPU oracle cannot
// reach; the tcgen05 path is the fast one.
//
// One CTA = 32 particle rows, 512 threads, on the shared fp32 tile engine (dmip_tile.cuh): activations live in
// shared memory, transposed and double-buffered; every layer is one tile_gemm against the weights, pre-transposed
// to [k][n] in the caller's workspace, followed by one bias + activation pass.  The whole S-step loop of a tile runs
// inside one launch (state in `out`, which only its owner thread touches).
//
// Reference code replaced: models/diffusion.py:27-46,158-180; sdes.py:21-49,77-87; nets.py:17-57,143-157.
#include "dmip_common.h"
#include "dmip_rng.cuh"
#include "dmip_sde.cuh"
#include "dmip_tile.cuh"

namespace dmip {

namespace {

constexpr int kMaxDpsX = 128;   // DPS: rows of the prior-output stash behind the weight slabs (227 KB in all)

struct NetDev {
  int n_layers, in_dim, out_dim;
  int width[DMIP_MAX_LAYERS];
  const float* Wt[DMIP_MAX_LAYERS];  // transposed [k][n]
  const float* b[DMIP_MAX_LAYERS];
};

struct F32Params {
  int mode, variant, n_nets;  // mode 0 sampler, 1 forward
  NetDev net[2];              // DPS: net[0] = prior (MLP2 on [x,t]), net[1] = likelihood (MLP on [x,y,t])
  int xdim, ydim, n_obs, tiles_per_obs, S;
  long long n_per_obs, n_tiles;
  float T, bmin, bmax, mean, std, delta, sqrt_delta;   // bmin / bmax: beta range (VP) or sigma range (VE)
  int sde_kind, n_corr;
  float snr;
  const float* y;
  float* out;
  int rng_mode;
  unsigned long long seed, gidx_base;
  const float* x0;
  const float* noise;
  const float* ynoise;
  const float* fx;
  const float* fcond;
  const float* ft;
  int fx_dim, fcond_dim;
};

__global__ void __launch_bounds__(kThreadsL, 1) k_f32_mlp(const __grid_constant__ F32Params P) {
  extern __shared__ __align__(16) float smem[];
  float* buf0 = smem;
  float* buf1 = smem + kMaxW * kLd;
  float* wbuf = buf1 + kMaxW * kLd;     // weight slabs of the staged GEMM
  float* stash = wbuf + kWbufFloats;    // DPS only: [xdim][kLd] prior output
  const int t = threadIdx.x, lane = t & 31;
  const long long n_total = static_cast<long long>(P.n_obs) * P.n_per_obs;

  // the net on the 32 rows whose inputs sit in buf0 ([in_dim][kLd]); returns the buffer holding the outputs
  // ([out_dim][kLd]).  Ends with __syncthreads().
  auto eval = [&](const NetDev& net) -> float* {
    float* in = buf0;
    float* out = buf1;
    int K = net.in_dim;
    for (int l = 0; l < net.n_layers; ++l) {
      const int N = net.width[l];
      tile_gemm(in, out, net.Wt[l], K, N, wbuf);
      const bool last = (l == net.n_layers - 1);
      for (int idx = t; idx < N * kRows; idx += kThreadsL) {   // a warp = one unit n, lane = row
        const int n = idx >> 5;
        float v = out[n * kLd + lane] + net.b[l][n];
        if (!last) {
          v = tanhf(v);
          if (l == 0) v = tanhf(v);  // the 'act' module registered twice (nets.py:25-30, SURVEY.md Q1)
        }
        out[n * kLd + lane] = v;
      }
      __syncthreads();
      float* tmp = in; in = out; out = tmp;
      K = N;
    }
    return in;
  };

  for (long long tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x) {
    const int obs = static_cast<int>(tile / P.tiles_per_obs);
    const long long prow0 = (tile % P.tiles_per_obs) * kRows;
    const long long grow0 = static_cast<long long>(obs) * P.n_per_obs + prow0;

    if (P.mode == 1) {
      // ---------------- forward: cat[x, cond, t] -> net -> out
      const NetDev& net = P.net[0];
      for (int idx = t; idx < kRows * net.in_dim; idx += kThreadsL) {
        const int k = idx / kRows, r = idx % kRows;
        float v = 0.f;
        if (prow0 + r < P.n_per_obs) {
          const long long g = grow0 + r;
          if (k < P.fx_dim) v = P.fx[g * P.fx_dim + k];
          else if (k < P.fx_dim + P.fcond_dim) v = P.fcond[g * P.fcond_dim + (k - P.fx_dim)];
          else v = P.ft[g];
        }
        buf0[k * kLd + r] = v;
      }
      __syncthreads();
      const float* res = eval(net);
      for (int idx = t; idx < kRows * net.out_dim; idx += kThreadsL) {
        const int r = idx / net.out_dim, j = idx % net.out_dim;
        if (prow0 + r < P.n_per_obs) P.out[(grow0 + r) * net.out_dim + j] = res[j * kLd + r];
      }
      __syncthreads();
      continue;
    }

    // ---------------- sampler
    const int nq = (P.xdim + 3) >> 2;
    for (int idx = t; idx < kRows * nq; idx += kThreadsL) {  // x0 = randn * std + mean (models/diffusion.py:32-33)
      const int r = idx % kRows, q = idx / kRows;
      if (prow0 + r >= P.n_per_obs) continue;
      const long long g = grow0 + r;
      float z[4];
      if (P.rng_mode == DMIP_RNG_PHILOX) philox_normal4(P.gidx_base + g, kPhiloxStepInit, kStreamState, q, P.seed, z);
      for (int e = 0; e < 4 && q * 4 + e < P.xdim; ++e) {
        const int j = q * 4 + e;
        const float zz = P.rng_mode == DMIP_RNG_PHILOX ? z[e] : P.x0[g * P.xdim + j];
        P.out[g * P.xdim + j] = zz * P.std + P.mean;
      }
    }
    __syncthreads();

    const SdeSched sch = {P.sde_kind, P.S, P.n_corr, P.T, P.bmin, P.bmax, P.snr, P.delta, P.sqrt_delta};
    const int n_sub = P.S * (1 + P.n_corr);        // sub-steps: predictor + correctors (dmip_sde.cuh)
    for (int step = 0; step < n_sub; ++step) {
      const SdeCoef co = sde_coef<false>(sch, step, P.variant == DMIP_DPS);
      const float tau = co.tau;
      const float sb = co.g;                       // g(tau): sqrt(beta) for the VP-SDE
      const float* res = nullptr;
      for (int p = 0; p < P.n_nets; ++p) {
        const NetDev& net = P.net[p];
        // ---- input rows: [x, (y | y_t), tau]   (nets.py:33 / :55)
        const bool with_y = !(P.variant == DMIP_DPS && p == 0);
        for (int idx = t; idx < kRows * net.in_dim; idx += kThreadsL) {
          const int k = idx / kRows, r = idx % kRows;
          float v = 0.f;
          if (prow0 + r < P.n_per_obs) {
            const long long g = grow0 + r;
            if (k < P.xdim) v = P.out[g * P.xdim + k];
            else if (with_y && k < P.xdim + P.ydim) {
              const int jj = k - P.xdim;
              v = P.y[obs * P.ydim + jj];
              if (P.variant == DMIP_CDIFFE) {
                // y_t = eta * std(tau) + alpha(tau) y   (sdes.py:37-49 <- models/diffusion.py:172)
                float g2u, alpha, var;
                sde_terms<false>(sch, tau, g2u, alpha, var);
                float eta;
                if (P.rng_mode == DMIP_RNG_PHILOX) {
                  float z[4];
                  philox_normal4(P.gidx_base + g, step, kStreamObs, jj >> 2, P.seed, z);
                  eta = z[jj & 3];
                } else {
                  eta = P.ynoise[(static_cast<long long>(step) * n_total + g) * P.ydim + jj];
                }
                v = eta * sqrtf(var) + alpha * v;
              }
            } else v = tau;
          }
          buf0[k * kLd + r] = v;
        }
        __syncthreads();
        res = eval(net);
        if (P.n_nets == 2 && p == 0) {
          for (int idx = t; idx < kRows * P.xdim; idx += kThreadsL) {
            const int j = idx / kRows, r = idx % kRows;
            stash[j * kLd + r] = res[j * kLd + r];
          }
          __syncthreads();
        }
      }
      // ---- Euler–Maruyama update (models/diffusion.py:40-42; sdes.py:77-79,86-87)
      for (int idx = t; idx < kRows * nq; idx += kThreadsL) {
        const int r = idx % kRows, q = idx / kRows;
        if (prow0 + r >= P.n_per_obs) continue;
        const long long g = grow0 + r;
        float z[4];
        if (P.rng_mode == DMIP_RNG_PHILOX) philox_normal4(P.gidx_base + g, step, kStreamState, q, P.seed, z);
        for (int e = 0; e < 4 && q * 4 + e < P.xdim; ++e) {
          const int j = q * 4 + e;
          float a = res[j * kLd + r];
          if (P.variant == DMIP_DPS) a = sb * (stash[j * kLd + r] + a);  // PosteriorScore: g * (prior + lik)
          const float x = P.out[g * P.xdim + j];
          const float eps = P.rng_mode == DMIP_RNG_PHILOX
                                ? z[e]
                                : P.noise[(static_cast<long long>(step) * n_total + g) * P.xdim + j];
          if (!co.corrector) {
            const float mu = sb * a + co.fx * x;              // g a - f   (sdes.py:77-79; fx = beta / 2 for VP, 0 for VE)
            P.out[g * P.xdim + j] = x + P.delta * mu + (P.sqrt_delta * sb) * eps;
          } else {
            // Langevin corrector: x += e score + sqrt(2 e) z with score = a / g (a already carries g for DPS: sb * sum)
            const float e = 0.5f * co.ke * co.ke;
            P.out[g * P.xdim + j] = x + (e / sb) * a + co.ke * eps;
          }
        }
      }
      __syncthreads();
    }
  }
}

int launch_f32(const F32Params& P, cudaStream_t s) {
  static int n_sm = 0;
  static bool ready[64] = {};   // cudaFuncSetAttribute is per device
  // buf0 | buf1 | weight slabs | DPS stash: 2 x 73 728 + 66 560 + 18 432 B at most, the opt-in limit per block
  const int smem_max = (2 * kMaxW * kLd + kWbufFloats + kMaxDpsX * kLd) * 4;
  const int smem = (2 * kMaxW * kLd + kWbufFloats + (P.n_nets == 2 ? P.xdim * kLd : 0)) * 4;
  int dev = 0;
  DMIP_CHECK_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || !ready[dev]) {
    DMIP_CHECK_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
    DMIP_CHECK_CUDA(cudaFuncSetAttribute(k_f32_mlp, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
    if (dev >= 0 && dev < 64) ready[dev] = true;
  }
  const long long grid = P.n_tiles < n_sm ? P.n_tiles : n_sm;
  if (grid <= 0) return DMIP_OK;
  k_f32_mlp<<<static_cast<unsigned>(grid), kThreadsL, smem, s>>>(P);
  DMIP_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return DMIP_OK;
}

}  // namespace

size_t sampler_f32_workspace(const DmipSampler* d) {
  return tile_net_bytes(d->net) + (d->variant == DMIP_DPS ? tile_net_bytes(d->net2) : 0);
}
size_t forward_f32_workspace(const DmipForward* d) { return tile_net_bytes(d->net); }

// after check_sampler (dmip_api.cu), which matches the nets' in / out dims to the descriptor
int launch_sampler_f32(const DmipSampler* d, cudaStream_t s) {
  F32Params P = {};
  P.mode = 0;
  P.variant = d->variant;
  const bool dps = d->variant == DMIP_DPS;
  DMIP_REQUIRE(!dps || d->xdim <= kMaxDpsX, "DPS fp32 sampler supports xdim <= %d", kMaxDpsX);
  P.n_nets = dps ? 2 : 1;
  const DmipMlp* nets[2] = {dps ? &d->net2 : &d->net, &d->net};   // DPS: net[0] = prior, net[1] = likelihood
  const char* names[2] = {dps ? "prior_net" : "net", "likelihood_net"};
  int rc;
  for (int p = 0; p < P.n_nets; ++p)
    if ((rc = tile_net_check(*nets[p], nets[p]->in_dim, names[p]))) return rc;
  uint8_t* ws = static_cast<uint8_t*>(d->workspace);
  for (int p = 0; p < P.n_nets; ++p) {
    if ((rc = tile_net_stage(*nets[p], ws, &P.net[p], s))) return rc;
    ws += tile_net_bytes(*nets[p]);
  }
  P.xdim = d->xdim;
  P.ydim = d->ydim;
  P.n_obs = d->n_obs;
  P.n_per_obs = d->n_per_obs;
  P.tiles_per_obs = static_cast<int>((d->n_per_obs + kRows - 1) / kRows);
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
  const double delta = static_cast<double>(d->T) / d->num_steps;
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
  return launch_f32(P, s);
}

int launch_forward_f32(const DmipForward* d, cudaStream_t s) {
  F32Params P = {};
  P.mode = 1;
  P.n_nets = 1;
  int rc;
  if ((rc = tile_net_check(d->net, d->net.in_dim, "net"))) return rc;
  if ((rc = tile_net_stage(d->net, d->workspace, &P.net[0], s))) return rc;
  P.n_obs = 1;
  P.n_per_obs = d->n;
  P.tiles_per_obs = static_cast<int>((d->n + kRows - 1) / kRows);
  P.n_tiles = P.tiles_per_obs;
  P.S = 1;
  P.out = d->out;
  P.fx = d->x;
  P.fcond = d->cond;
  P.ft = d->t;
  P.fx_dim = d->x_dim;
  P.fcond_dim = d->cond_dim;
  return launch_f32(P, s);
}

}  // namespace dmip
