// dmip_f32.cu — the fp32 (FFMA) path: the same fused sampler / forward as dmip_tc.cu for ANY layer widths
// (<= 512) and to fp32 round-off of the reference (accurate tanhf, no operand rounding).  It is the strict-
// parity mode of the product and the GPU-side cross-check of the tcgen05 path at sizes the CPU oracle cannot
// reach; the tcgen05 path is the fast one.
//
// One CTA = 32 particle rows, 256 threads.  Activations live in shared memory, transposed ([k][row], row
// stride 36 floats) and double-buffered; every layer is a 32 x N x K register-tiled GEMM (8 rows x 8 columns
// per thread) reading the weights, pre-transposed to [k][n] in the caller's workspace, straight from L2/L1.
// The whole S-step loop of a tile runs inside one launch (state in `out`, which only its owner thread touches).
//
// Reference code replaced: models/diffusion.py:27-46,158-180; sdes.py:21-49,77-87; nets.py:17-57,143-157.
#include "dmip_common.h"
#include "dmip_rng.cuh"
#include "dmip_sde.cuh"

namespace dmip {

namespace {

constexpr int kRows = 32;
constexpr int kLd = 36;       // row stride of the transposed activation buffers
constexpr int kMaxW = 512;    // max layer width / input width
constexpr int kThreadsF = 256;

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

// Evaluate the net on the 32 rows whose inputs sit in buf0 ([in_dim][kLd]).  Returns the buffer holding the
// outputs ([out_dim][kLd]).  All 256 threads participate; ends with __syncthreads().
__device__ float* mlp_eval(const NetDev& net, float* buf0, float* buf1) {
  const int t = threadIdx.x;
  const int rg = t >> 6, ng = t & 63;
  float* in = buf0;
  float* outb = buf1;
  int K = net.in_dim;
  for (int l = 0; l < net.n_layers; ++l) {
    const int N = net.width[l];
    const float* __restrict__ Wt = net.Wt[l];
    float acc[8][8];
#pragma unroll
    for (int r = 0; r < 8; ++r)
#pragma unroll
      for (int i = 0; i < 8; ++i) acc[r][i] = 0.f;
    const int ncols = (N - ng + 63) >> 6;  // number of valid columns of this thread (n = ng + 64 i < N)
    if (ncols > 0) {
      for (int k = 0; k < K; ++k) {
        const float4 a0 = *reinterpret_cast<const float4*>(in + k * kLd + rg * 8);
        const float4 a1 = *reinterpret_cast<const float4*>(in + k * kLd + rg * 8 + 4);
        const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        float w[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) w[i] = (i < ncols) ? __ldg(Wt + static_cast<size_t>(k) * N + ng + 64 * i) : 0.f;
#pragma unroll
        for (int r = 0; r < 8; ++r)
#pragma unroll
          for (int i = 0; i < 8; ++i) acc[r][i] = fmaf(a[r], w[i], acc[r][i]);
      }
    }
    const bool last = (l == net.n_layers - 1);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int n = ng + 64 * i;
      if (n < N) {
        const float bb = net.b[l][n];
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          float v = acc[r][i] + bb;
          if (!last) {
            v = tanhf(v);
            if (l == 0) v = tanhf(v);  // the 'act' module registered twice (nets.py:25-30, SURVEY.md Q1)
          }
          outb[n * kLd + rg * 8 + r] = v;
        }
      }
    }
    __syncthreads();
    float* tmp = in;
    in = outb;
    outb = tmp;
    K = N;
  }
  return in;
}

__global__ void __launch_bounds__(kThreadsF, 1) k_f32_mlp(const __grid_constant__ F32Params P) {
  extern __shared__ float smemf[];
  float* buf0 = smemf;
  float* buf1 = smemf + kMaxW * kLd;
  float* stash = buf1 + kMaxW * kLd;  // [128][kLd] DPS prior output
  const int t = threadIdx.x;
  const long long n_total = static_cast<long long>(P.n_obs) * P.n_per_obs;
  const float dbeta = P.bmax - P.bmin;

  for (long long tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x) {
    const int obs = static_cast<int>(tile / P.tiles_per_obs);
    const long long prow0 = (tile % P.tiles_per_obs) * kRows;
    const long long grow0 = static_cast<long long>(obs) * P.n_per_obs + prow0;

    if (P.mode == 1) {
      // ---------------- forward: cat[x, cond, t] -> net -> out
      const NetDev& net = P.net[0];
      for (int idx = t; idx < kRows * net.in_dim; idx += kThreadsF) {
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
      const float* res = mlp_eval(net, buf0, buf1);
      for (int idx = t; idx < kRows * net.out_dim; idx += kThreadsF) {
        const int r = idx / net.out_dim, j = idx % net.out_dim;
        if (prow0 + r < P.n_per_obs) P.out[(grow0 + r) * net.out_dim + j] = res[j * kLd + r];
      }
      __syncthreads();
      continue;
    }

    // ---------------- sampler
    const int nq = (P.xdim + 3) >> 2;
    for (int idx = t; idx < kRows * nq; idx += kThreadsF) {  // x0 = randn * std + mean (models/diffusion.py:32-33)
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
        for (int idx = t; idx < kRows * net.in_dim; idx += kThreadsF) {
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
                float alpha, sd;
                if (P.sde_kind == kSdeVE) {
                  float g2u, var;
                  sde_terms<false>(sch, tau, g2u, alpha, var);
                  sd = sqrtf(var);
                } else {
                  alpha = expf(-0.25f * tau * tau * dbeta - 0.5f * tau * P.bmin);
                  sd = sqrtf(1.0f - expf(-0.5f * tau * tau * dbeta - tau * P.bmin));
                }
                float eta;
                if (P.rng_mode == DMIP_RNG_PHILOX) {
                  float z[4];
                  philox_normal4(P.gidx_base + g, step, kStreamObs, jj >> 2, P.seed, z);
                  eta = z[jj & 3];
                } else {
                  eta = P.ynoise[(static_cast<long long>(step) * n_total + g) * P.ydim + jj];
                }
                v = eta * sd + alpha * v;
              }
            } else v = tau;
          }
          buf0[k * kLd + r] = v;
        }
        __syncthreads();
        res = mlp_eval(net, buf0, buf1);
        if (P.n_nets == 2 && p == 0) {
          for (int idx = t; idx < kRows * P.xdim; idx += kThreadsF) {
            const int j = idx / kRows, r = idx % kRows;
            stash[j * kLd + r] = res[j * kLd + r];
          }
          __syncthreads();
        }
      }
      // ---- Euler–Maruyama update (models/diffusion.py:40-42; sdes.py:77-79,86-87)
      for (int idx = t; idx < kRows * nq; idx += kThreadsF) {
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

__global__ void k_transpose(const float* __restrict__ W, float* __restrict__ Wt, int rows, int cols) {
  // W (rows, cols) -> Wt (cols, rows)
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

size_t net_ws_floats(const DmipMlp* net) {
  size_t n = 0;
  int k = net->in_dim;
  // sized before check_net() refuses a bad descriptor: read no slot past width[DMIP_MAX_LAYERS - 1]
  for (int l = 0; l < net->n_layers && l < DMIP_MAX_LAYERS; ++l) {
    if (k < 0 || net->width[l] < 0) return 0;
    n += static_cast<size_t>(k) * net->width[l];
    k = net->width[l];
  }
  return (n + 3) & ~size_t(3);
}

int check_net(const DmipMlp* net) {
  DMIP_REQUIRE(net->n_layers >= 2 && net->n_layers <= DMIP_MAX_LAYERS, "n_layers %d out of range", net->n_layers);
  DMIP_REQUIRE(net->in_dim >= 1 && net->in_dim <= kMaxW, "in_dim %d out of range (max %d)", net->in_dim, kMaxW);
  for (int l = 0; l < net->n_layers; ++l) {
    DMIP_REQUIRE(net->width[l] >= 1 && net->width[l] <= kMaxW, "layer %d width %d out of range (max %d)", l,
                 net->width[l], kMaxW);
    DMIP_REQUIRE(net->W[l] && net->b[l], "layer %d has a NULL pointer", l);
  }
  DMIP_REQUIRE(net->width[net->n_layers - 1] == net->out_dim, "last layer width != out_dim");
  return DMIP_OK;
}

int prep_net(const DmipMlp* net, float* ws, NetDev* o, cudaStream_t s) {
  int rc = check_net(net);
  if (rc) return rc;
  o->n_layers = net->n_layers;
  o->in_dim = net->in_dim;
  o->out_dim = net->out_dim;
  int k = net->in_dim;
  for (int l = 0; l < net->n_layers; ++l) {
    const int n = net->width[l];
    o->width[l] = n;
    o->Wt[l] = ws;
    o->b[l] = net->b[l];
    dim3 grid(ceil_div(k, 32), ceil_div(n, 32)), block(32, 8);
    k_transpose<<<grid, block, 0, s>>>(net->W[l], ws, n, k);
    DMIP_CHECK_CUDA(cudaGetLastError());
    count_launch();
    ws += static_cast<size_t>(k) * n;
    k = n;
  }
  return DMIP_OK;
}

int launch_f32(const F32Params& P, cudaStream_t s) {
  static int n_sm = 0;
  static bool ready[64] = {};   // cudaFuncSetAttribute is per device
  const int smem = (2 * kMaxW + 128) * kLd * 4;
  int dev = 0;
  DMIP_CHECK_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || !ready[dev]) {
    DMIP_CHECK_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
    DMIP_CHECK_CUDA(cudaFuncSetAttribute(k_f32_mlp, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    if (dev >= 0 && dev < 64) ready[dev] = true;
  }
  const long long grid = P.n_tiles < n_sm ? P.n_tiles : n_sm;
  if (grid <= 0) return DMIP_OK;
  k_f32_mlp<<<static_cast<unsigned>(grid), kThreadsF, smem, s>>>(P);
  DMIP_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return DMIP_OK;
}

}  // namespace

size_t sampler_f32_workspace(const DmipSampler* d) {
  size_t n = net_ws_floats(&d->net);
  if (d->variant == DMIP_DPS) n += net_ws_floats(&d->net2);
  return n * 4;
}
size_t forward_f32_workspace(const DmipForward* d) { return net_ws_floats(&d->net) * 4; }

int launch_sampler_f32(const DmipSampler* d, cudaStream_t s) {
  F32Params P = {};
  P.mode = 0;
  P.variant = d->variant;
  DMIP_REQUIRE(d->workspace && d->workspace_bytes >= sampler_f32_workspace(d), "workspace too small: need %zu bytes",
               sampler_f32_workspace(d));
  float* ws = static_cast<float*>(d->workspace);
  int rc;
  if (d->variant == DMIP_DPS) {
    P.n_nets = 2;
    DMIP_REQUIRE(d->xdim <= 128, "DPS fp32 sampler supports xdim <= 128");
    DMIP_REQUIRE(d->net2.in_dim == d->xdim + 1 && d->net2.out_dim == d->xdim, "prior_net must map [x,t] -> x");
    DMIP_REQUIRE(d->net.in_dim == d->xdim + d->ydim + 1 && d->net.out_dim == d->xdim,
                 "likelihood_net must map [x,y,t] -> x");
    if ((rc = prep_net(&d->net2, ws, &P.net[0], s))) return rc;
    ws += net_ws_floats(&d->net2);
    if ((rc = prep_net(&d->net, ws, &P.net[1], s))) return rc;
  } else {
    P.n_nets = 1;
    DMIP_REQUIRE(d->net.in_dim == d->xdim + d->ydim + 1, "net.in_dim must be xdim+ydim+1");
    DMIP_REQUIRE(d->net.out_dim >= d->xdim, "net.out_dim must be >= xdim");
    if ((rc = prep_net(&d->net, ws, &P.net[0], s))) return rc;
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
  DMIP_REQUIRE(d->workspace && d->workspace_bytes >= forward_f32_workspace(d), "workspace too small: need %zu bytes",
               forward_f32_workspace(d));
  int rc;
  if ((rc = prep_net(&d->net, static_cast<float*>(d->workspace), &P.net[0], s))) return rc;
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
