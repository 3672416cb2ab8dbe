// dmip_loss.cu — fused score-training losses, forward + backward, fp32 (K2 DSM, K3 PINN / Score-FPE, DSM_PDE).
//
// Replaces, per training batch: VariancePreservingSDE.sample (sdes.py:37-49), the net evaluations, DSMLoss
// (losses.py:49-52), ScoreFPELoss with exact divergence (losses.py:77-98: 2d+1 autograd double-backward passes),
// ConditionalScoreFPELoss (losses.py:116-124), DSM_PDELoss (losses.py:143-164), PINNLoss (losses.py:214-242) and
// the loss.backward() through that double-backward graph (models/diffusion.py:100-102).
//
// Method (SURVEY.md App. A.4/A.5): forward-mode jets instead of reverse-over-reverse autograd.  Every sample is
// expanded into "streams" that share the net's weights and therefore ride the same GEMMs as extra rows:
//     P   primal at [z_t, cond, t]            I   primal at [x, y, 0]            (PINN initial condition)
//     T   tangent along (dz_t/dt, 0, 1)       S_k tangents along e_k             Q_ik second-order pairs (i <= k)
// ds/dt is the TOTAL derivative along z_t(t) at fixed eps (Q8); grad_x [div s + |s|^2 + x.s] is a constant in the
// backward pass (Q9); the (B,)+(B,1) broadcast of the reference means mean(loss) = mean(dsm)+mean(ic)+mean(pde) (Q10).
// Parameter gradients flow through P, I and T only; the T adjoint couples back into P through phi' and phi''.
//
// Three kernels: k_jets_fwd (one CTA = 32 stream-rows: GEMM per layer + jet activation in shared memory, per-sample
// loss and top adjoints), k_jets_bwd (adjoint rows back through the layers), k_wgrad (dW_l = ADJ_l^T IN_l, split-K).
#include <stdlib.h>
#include <string.h>

#include "dmip_common.h"
#include "dmip_jets.cuh"
#include "dmip_tcl.h"
#include "dmip_tile.cuh"

namespace dmip {

namespace {

constexpr int kMaxD = 4;   // exact Score-FPE: state dimension of the diffused variable (d(d+1)/2 second-order streams)

// the problem (dmip_common.h: LossProblem, shared with the tcgen05 kernels), the net, the streams and the workspace
struct LossDev : LossProblem {
  int in_dim, out_dim, n_layers;
  int width[DMIP_MAX_LAYERS];
  const float* W[DMIP_MAX_LAYERS];    // original (out,in)
  const float* Wt[DMIP_MAX_LAYERS];   // transposed (in,out)
  const float* b[DMIP_MAX_LAYERS];
  int has_I, has_T, has_S, has_Q;     // stream groups present
  int n_streams, spt;                 // streams per sample, samples per tile
  int n_adj;                          // adjoint streams per sample: P [, I] [, T]
  int n_tan;                          // spatial tangent streams: d (directions e_k) or 1 (Hutchinson probe v)
  const float* hutch_v;               // post=3, Hutchinson: probe v (B,d); NULL = exact (e_k)
  float* tan_z[DMIP_MAX_LAYERS];      // post=3: TAN_l [B][n_tan][N_l] pre-activation spatial tangents of hidden layer l
  float* in_rows[DMIP_MAX_LAYERS];    // IN_l  [B*n_adj][K_l]   inputs of layer l for the adjoint streams
  float* adj_rows[DMIP_MAX_LAYERS];   // ADJ_l [B*n_adj][N_l]   adjoints of layer l pre-activations
  float* zdt[DMIP_MAX_LAYERS];        // ZDT_l [B][N_l]         pre-activation time tangent of hidden layer l
  float* abar;                        // [B*n_adj][out_dim]     adjoints of the net outputs
};

// activation jets: value h, first and second derivative of phi at pre-activation z (layer 0: tanh(tanh), else tanh)
__device__ __forceinline__ void act_jet(float z, bool first, float& h, float& p1, float& p2) {
  if (first) {
    const float u = tanhf(z);
    h = tanhf(u);
    p1 = (1.f - h * h) * (1.f - u * u);
    p2 = p1 * (-2.f * h * (1.f - u * u) - 2.f * u);
  } else {
    h = tanhf(z);
    p1 = 1.f - h * h;
    p2 = -2.f * h * p1;
  }
}

// phi', phi'' of a hidden layer from its stored output h (layer 0: h = tanh(u), u = atanh(h), |h| < tanh(1))
__device__ __forceinline__ void dphi_from_h(float h, bool first, float& p1, float& p2) {
  if (first) {
    const float u = atanhf(h);
    p1 = (1.f - h * h) * (1.f - u * u);
    p2 = p1 * (-2.f * h * (1.f - u * u) - 2.f * u);
  } else {
    p1 = 1.f - h * h;
    p2 = -2.f * h * p1;
  }
}

// stream layout of a pass (dmip_jets.cuh), at run time
struct Streams {
  int kI, kT, sI, sT, sS, sQ, NADJ;
};

// staged net outputs of one sample in k_jets_fwd: o[component * kLd + stream], output bias b added on read
struct FfmaOuts {
  const float* o;
  const float* b;
  __device__ __forceinline__ float primal(int s, int c) const { return o[c * kLd + s] + b[c]; }
  __device__ __forceinline__ float tangent(int s, int c) const { return o[c * kLd + s]; }
};

// ------------------------------------------------------------------------------------------------ forward
__global__ void __launch_bounds__(kThreadsL, 1) k_jets_fwd(const __grid_constant__ LossDev P) {
  extern __shared__ __align__(16) float smem[];
  float* buf0 = smem;
  float* buf1 = smem + kMaxW * kLd;
  float* wbuf = buf1 + kMaxW * kLd;   // weight slabs of the staged GEMM
  __shared__ float red[4];
  const int t = threadIdx.x;
  const int ns = P.n_streams, spt = P.spt, d = P.d;
  const int sS = 1 + P.has_I + P.has_T;
  const Streams S = {P.has_I, P.has_T, 1, 1 + P.has_I, sS, sS + (P.has_S ? P.n_tan : 0), P.n_adj};
  const long long n_tiles = (P.B + spt - 1) / spt;

  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long s0 = tile * spt;
    if (t < 4) red[t] = 0.f;
    // ---- layer-0 input rows
    for (int idx = t; idx < kRows * P.in_dim; idx += kThreadsL) {
      const int k = idx / kRows, r = idx % kRows;
      const int sl = r / ns, st = r % ns;
      const long long smp = s0 + sl;
      float v = 0.f;
      if (sl < spt && smp < P.B) {
        if (P.hutch_v && st >= S.sS && st < S.sQ)
          v = (k < d) ? P.hutch_v[smp * d + k] : 0.f;          // Hutchinson probe   (losses.py:28-40)
        else
          v = jet_input(P, S, sample_vp(P, smp), smp, st, k);
        // inputs of layer 0 for the adjoint streams (wgrad operands)
        const int aidx = (st == 0) ? 0 : (P.has_I && st == S.sI) ? 1 : (P.has_T && st == S.sT) ? (1 + P.has_I) : -1;
        if (aidx >= 0) P.in_rows[0][(smp * P.n_adj + aidx) * P.in_dim + k] = v;
      }
      buf0[k * kLd + r] = v;
    }
    __syncthreads();

    float* in = buf0;
    float* out = buf1;
    int K = P.in_dim;
    for (int l = 0; l < P.n_layers; ++l) {
      const int N = P.width[l];
      tile_gemm(in, out, P.Wt[l], K, N, wbuf);
      const bool last = (l == P.n_layers - 1);
      if (!last) {
        // ---- jet activation, in place: one (column, sample) pair per thread iteration
        for (int idx = t; idx < N * spt; idx += kThreadsL) {
          const int n = idx % N, sl = idx / N;
          const long long smp = s0 + sl;
          float* col = out + n * kLd + sl * ns;
          const float bias = P.b[l][n];
          float h, p1, p2;
          act_jet(col[0] + bias, l == 0, h, p1, p2);
          const bool live = smp < P.B;
          if (live) P.in_rows[l + 1][(smp * P.n_adj + 0) * N + n] = h;
          col[0] = h;
          if (P.has_I) {
            float hi, q1, q2;
            act_jet(col[S.sI] + bias, l == 0, hi, q1, q2);
            col[S.sI] = hi;
            if (live) P.in_rows[l + 1][(smp * P.n_adj + 1) * N + n] = hi;
          }
          if (P.has_T) {
            const float zd = col[S.sT];
            const float hd = p1 * zd;
            col[S.sT] = hd;
            if (live) {
              P.zdt[l][smp * N + n] = zd;
              P.in_rows[l + 1][(smp * P.n_adj + 1 + P.has_I) * N + n] = hd;
            }
          }
          if (P.post == 3) {
            for (int k = 0; k < P.n_tan; ++k) {
              const float zs = col[S.sS + k];
              if (live) P.tan_z[l][(smp * P.n_tan + k) * N + n] = zs;
              col[S.sS + k] = p1 * zs;
            }
          } else if (P.has_S) {
            float zs[kMaxD];
#pragma unroll
            for (int k = 0; k < kMaxD; ++k)
              if (k < d) zs[k] = col[S.sS + k];
            if (P.has_Q) {
#pragma unroll
              for (int i = 0; i < kMaxD; ++i)
#pragma unroll
                for (int k = i; k < kMaxD; ++k)
                  if (k < d) {
                    const int q = S.sQ + q_index(i, k, d);
                    col[q] = p1 * col[q] + p2 * zs[i] * zs[k];
                  }
            }
#pragma unroll
            for (int k = 0; k < kMaxD; ++k)
              if (k < d) col[S.sS + k] = p1 * zs[k];
          }
        }
        __syncthreads();
      }
      float* tmp = in;
      in = out;
      out = tmp;
      K = N;
    }

    if (P.post == 3) {
      // ---- grad_x pass: seeds of the reverse sweep for phi = div s + |s|^2 + x.s  (losses.py:88-90), with
      // div s = sum_k (S_k)_k / sqrt(beta) (exact) or v.(J v) / sqrt(beta) (Hutchinson):
      //   abar_P[j] = 2 a_j / beta + z_t[j] / sqrt(beta),  abar_Sk[j] = dir_k[j] / sqrt(beta);  direct term a_k / sqrt(beta)
      const int L = P.n_layers - 1, od = P.out_dim, na = 1 + P.n_tan;
      for (int idx = t; idx < spt * na * od; idx += kThreadsL) {
        const int j = idx % od, st = (idx / od) % na, sl = idx / (od * na);
        const long long smp = s0 + sl;
        if (smp >= P.B) continue;
        const SampleVp vp = sample_vp(P, smp);
        const float sb = sqrtf(vp.beta);
        float v;
        if (st == 0) {
          const float a = in[j * kLd + sl * ns] + P.b[L][j];
          const float zt = P.eps[smp * d + j] * vp.sd + vp.alpha * state0(P, smp, j);
          v = 2.f * a / vp.beta + zt / sb;
          P.gradx[smp * d + j] = a / sb;
        } else {
          const float dir = P.hutch_v ? P.hutch_v[smp * d + j] : (j == st - 1 ? 1.f : 0.f);
          v = dir / sb;
        }
        P.abar[(smp * na + st) * od + j] = v;
      }
      __syncthreads();
      continue;
    }
    // ---- loss terms and output adjoints, one (sample, output component) item per thread (`in` holds the raw
    // last-layer rows, dmip_jets.cuh: jet_loss_item); partial sums meet in red[] through warp shuffles
    {
      const int L = P.n_layers - 1, od = P.out_dim;
      const int n_items = spt * od;
      for (int base = 0; base < n_items; base += kThreadsL) {
        const int idx = base + t;
        const int sl = idx / od, j = idx - sl * od;
        const long long smp = s0 + sl;
        float l_dsm = 0.f, l_ic = 0.f, l_pde = 0.f;
        if (idx < n_items && smp < P.B)
          jet_loss_item(P, S, FfmaOuts{in + sl * ns, P.b[L]}, P.abar, od, smp, j, l_dsm, l_ic, l_pde);
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
    __syncthreads();
    if (t == 0) {
      atomicAdd(&P.losses[1], red[1] * P.inv_B);
      atomicAdd(&P.losses[2], red[2] * P.inv_B);
      atomicAdd(&P.losses[3], red[3] * P.inv_B);
      atomicAdd(&P.losses[0], ((P.kind == DMIP_LOSS_PINN2 ? 0.f : red[1]) + red[2] + red[3]) * P.inv_B);
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------ backward
// rows = (sample, adjoint stream); P and T rows of a sample are coupled through phi' and phi''.
__global__ void __launch_bounds__(kThreadsL, 1) k_jets_bwd(const __grid_constant__ LossDev P) {
  extern __shared__ __align__(16) float smem[];
  float* buf0 = smem;
  float* buf1 = smem + kMaxW * kLd;
  float* wbuf = buf1 + kMaxW * kLd;   // weight slabs of the staged GEMM
  const int t = threadIdx.x;
  const int na = P.n_adj;
  const int spt = kRows / na;
  const int aT = 1 + P.has_I;
  const long long n_tiles = (P.B + spt - 1) / spt;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long s0 = tile * spt;
    const int L = P.n_layers - 1;
    // adjoints of the outputs = adjoints of the last layer's pre-activations
    for (int idx = t; idx < kRows * P.out_dim; idx += kThreadsL) {
      const int n = idx / kRows, r = idx % kRows;
      const int sl = r / na, st = r % na;
      const long long smp = s0 + sl;
      float v = 0.f;
      if (sl < spt && smp < P.B) {
        v = P.abar[(smp * na + st) * P.out_dim + n];
        P.adj_rows[L][(smp * na + st) * P.out_dim + n] = v;
      }
      buf0[n * kLd + r] = v;
    }
    __syncthreads();
    float* in = buf0;
    float* out = buf1;
    for (int l = L; l >= 1; --l) {
      const int N = P.width[l], Kp = P.width[l - 1];
      tile_gemm(in, out, P.W[l], N, Kp, wbuf);      // hbar_{l-1}[k] = sum_n zbar_l[n] W_l[n][k]
      for (int idx = t; idx < Kp * spt; idx += kThreadsL) {
        const int k = idx % Kp, sl = idx / Kp;
        const long long smp = s0 + sl;
        if (smp >= P.B) continue;
        float* col = out + k * kLd + sl * na;
        float p1, p2;
        dphi_from_h(P.in_rows[l][(smp * na + 0) * Kp + k], l - 1 == 0, p1, p2);
        float zP = p1 * col[0];
        if (P.has_T) {
          const float hdbar = col[aT];
          zP += p2 * P.zdt[l - 1][smp * Kp + k] * hdbar;
          const float zT = p1 * hdbar;
          col[aT] = zT;
          P.adj_rows[l - 1][(smp * na + aT) * Kp + k] = zT;
        }
        col[0] = zP;
        P.adj_rows[l - 1][(smp * na + 0) * Kp + k] = zP;
        if (P.has_I) {
          float q1, q2;
          dphi_from_h(P.in_rows[l][(smp * na + 1) * Kp + k], l - 1 == 0, q1, q2);
          const float zI = q1 * col[1];
          col[1] = zI;
          P.adj_rows[l - 1][(smp * na + 1) * Kp + k] = zI;
        }
      }
      __syncthreads();
      float* tmp = in;
      in = out;
      out = tmp;
    }
  }
}

// ------------------------------------------------------------------------------------------------ grad_x (adjoint route)
// Reverse sweep through the (primal, spatial tangents) jet of the post=3 forward pass; rows = (sample, P | S_k).
// With hbar the adjoint of h and hdbar_k those of the tangents hd_k = phi'(z) zd_k:
//     zbar = phi' hbar + phi'' sum_k zd_k hdbar_k,     zdbar_k = phi' hdbar_k,
// and the gradient w.r.t. the diffused state is the first d columns of zbar_0 W_0.  Cost (2 + n_tan) net passes instead of
// the d(d+1)/2 second-order streams of the forward-only route: this is what makes d = 26 (CDiffE, scatterometry) and the
// Hutchinson estimator (n_tan = 1) affordable.  Nothing here carries a parameter gradient (grad_x is detached, Q9).
__global__ void __launch_bounds__(kThreadsL, 1) k_gradx_bwd(const __grid_constant__ LossDev P) {
  extern __shared__ __align__(16) float smem[];
  float* buf0 = smem;
  float* buf1 = smem + kMaxW * kLd;
  float* wbuf = buf1 + kMaxW * kLd;
  const int t = threadIdx.x;
  const int nt = P.n_tan, na = 1 + nt, d = P.d;
  const int spt = kRows / na;
  const long long n_tiles = (P.B + spt - 1) / spt;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long s0 = tile * spt;
    const int L = P.n_layers - 1;
    for (int idx = t; idx < kRows * P.out_dim; idx += kThreadsL) {
      const int n = idx / kRows, r = idx % kRows;
      const int sl = r / na, st = r % na;
      const long long smp = s0 + sl;
      buf0[n * kLd + r] = (sl < spt && smp < P.B) ? P.abar[(smp * na + st) * P.out_dim + n] : 0.f;
    }
    __syncthreads();
    float* in = buf0;
    float* out = buf1;
    for (int l = L; l >= 1; --l) {
      const int N = P.width[l], Kp = P.width[l - 1];
      tile_gemm(in, out, P.W[l], N, Kp, wbuf);
      for (int idx = t; idx < Kp * spt; idx += kThreadsL) {
        const int k = idx % Kp, sl = idx / Kp;
        const long long smp = s0 + sl;
        if (smp >= P.B) continue;
        float* col = out + k * kLd + sl * na;
        float p1, p2;
        dphi_from_h(P.in_rows[l][smp * Kp + k], l - 1 == 0, p1, p2);
        float cross = 0.f;
        for (int j = 0; j < nt; ++j) {
          const float hdbar = col[1 + j];
          cross = fmaf(P.tan_z[l - 1][(smp * nt + j) * Kp + k], hdbar, cross);
          col[1 + j] = p1 * hdbar;
        }
        col[0] = p1 * col[0] + p2 * cross;
      }
      __syncthreads();
      float* tmp = in;
      in = out;
      out = tmp;
    }
    tile_gemm(in, out, P.W[0], P.width[0], P.in_dim, wbuf);   // xbar[k] = sum_n zbar_0[n] W_0[n][k]
    for (int idx = t; idx < d * spt; idx += kThreadsL) {
      const int k = idx % d, sl = idx / d;
      const long long smp = s0 + sl;
      if (smp < P.B) P.gradx[smp * d + k] += out[k * kLd + sl * na];
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------ weight gradients
// dW[n][k] += sum_r ADJ[r][n] * IN[r][k]   (r over B*n_adj rows), db[n] += sum_{r: stream is P or I} ADJ[r][n].
// 128 x 128 output tile per CTA (256 threads, 8 x 8 outputs each, operands staged through double-buffered shared
// memory 8 rows at a time), split over row ranges (gridDim.z), fp32 atomics into the flat gradient buffer.
constexpr int kWgT = 128;   // tile edge
constexpr int kWgR = 8;     // rows per stage

__global__ void __launch_bounds__(256) k_wgrad(const float* __restrict__ adj, const float* __restrict__ inp, float* dW,
                                               float* db, long long rows, int N, int K, int n_adj, int bias_streams,
                                               long long rows_per_split) {
  __shared__ __align__(16) float sA[2][kWgR][kWgT];
  __shared__ __align__(16) float sI[2][kWgR][kWgT];
  const int n0 = blockIdx.y * kWgT, k0 = blockIdx.x * kWgT;
  const long long r_begin = static_cast<long long>(blockIdx.z) * rows_per_split;
  const long long r_end = min(rows, r_begin + rows_per_split);
  const int t = threadIdx.x;
  const int tx = t & 15, ty = t >> 4;          // outputs: n = n0 + ty*4 + {0..3} and + 64; k = k0 + tx*4 + {0..3} and + 64
  const int lr = t >> 5, lc = (t & 31) * 4;    // loader: row lr of the stage, columns lc .. lc+3
  const bool vecA = (N & 3) == 0, vecI = (K & 3) == 0;

  auto load = [&](const float* __restrict__ src, int ld, int c0, bool vec, long long r, float (&v)[4]) {
    v[0] = v[1] = v[2] = v[3] = 0.f;
    if (r < r_end) {
      const int c = c0 + lc;
      const float* p = src + r * ld + c;
      if (vec && c + 3 < ld) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(p));
        v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (c + e < ld) v[e] = __ldg(p + e);
      }
    }
  };

  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  float bsum[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) bsum[i] = 0.f;

  float va[4], vi[4];
  load(adj, N, n0, vecA, r_begin + lr, va);
  load(inp, K, k0, vecI, r_begin + lr, vi);
  *reinterpret_cast<float4*>(&sA[0][lr][lc]) = make_float4(va[0], va[1], va[2], va[3]);
  *reinterpret_cast<float4*>(&sI[0][lr][lc]) = make_float4(vi[0], vi[1], vi[2], vi[3]);
  __syncthreads();
  int cur = 0;
  for (long long r0 = r_begin; r0 < r_end; r0 += kWgR) {
    const bool more = r0 + kWgR < r_end;
    if (more) {   // global loads of the next stage fly while this stage is multiplied
      load(adj, N, n0, vecA, r0 + kWgR + lr, va);
      load(inp, K, k0, vecI, r0 + kWgR + lr, vi);
    }
#pragma unroll
    for (int rr = 0; rr < kWgR; ++rr) {
      const float4 a0 = *reinterpret_cast<const float4*>(&sA[cur][rr][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&sA[cur][rr][64 + ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&sI[cur][rr][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&sI[cur][rr][64 + tx * 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      if (blockIdx.x == 0 && tx == 0 && ((r0 + rr) % n_adj) < bias_streams) {
#pragma unroll
        for (int i = 0; i < 8; ++i) bsum[i] += a[i];
      }
    }
    if (more) {
      *reinterpret_cast<float4*>(&sA[cur ^ 1][lr][lc]) = make_float4(va[0], va[1], va[2], va[3]);
      *reinterpret_cast<float4*>(&sI[cur ^ 1][lr][lc]) = make_float4(vi[0], vi[1], vi[2], vi[3]);
    }
    __syncthreads();
    cur ^= 1;
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int n = n0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
    if (n >= N) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = k0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
      if (k < K) atomicAdd(&dW[static_cast<size_t>(n) * K + k], acc[i][j]);
    }
    if (blockIdx.x == 0 && tx == 0) atomicAdd(&db[n], bsum[i]);
  }
}



// Skinny weight gradient: one side of dW = ADJ^T IN has at most kSkinny columns (layer 0: K = in_dim = 5 ... 8; output
// layer: N = out_dim = 2 ... 8) — a 128 x 128 tile would waste 94 ... 98 % of its FMAs and ran 14x above the HBM time of
// reading the wide operand once.  Thread = 4 consecutive columns of the wide matrix (float4, coalesced), the narrow
// row is a broadcast load; a CTA walks a row range, 4 rows in flight; fp32 atomics at the end.
constexpr int kSkinny = 8;

template <bool kAdjWide>
__global__ void __launch_bounds__(128) k_wgrad_skinny(const float* __restrict__ adj, const float* __restrict__ inp, float* dW,
                                                      float* db, long long rows, int N, int K, int n_adj, int bias_streams,
                                                      long long rows_per_cta) {
  const int W = kAdjWide ? N : K, S = kAdjWide ? K : N;        // wide / narrow column counts
  const float* __restrict__ wide = kAdjWide ? adj : inp;
  const float* __restrict__ nar = kAdjWide ? inp : adj;
  const int c = (blockIdx.y * 128 + threadIdx.x) * 4;          // W % 4 == 0 (checked on the host)
  if (c >= W) return;
  const long long r0 = static_cast<long long>(blockIdx.x) * rows_per_cta;
  const long long r1 = min(rows, r0 + rows_per_cta);
  float acc[kSkinny][4];
#pragma unroll
  for (int j = 0; j < kSkinny; ++j) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
  float bs[4] = {0.f, 0.f, 0.f, 0.f};                          // bias sums: wide columns (kAdjWide) ...
  float bn[kSkinny];                                           // ... or narrow columns
#pragma unroll
  for (int j = 0; j < kSkinny; ++j) bn[j] = 0.f;
  for (long long r = r0; r < r1; r += 4) {
    float4 w[4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
      w[u] = (r + u < r1) ? __ldg(reinterpret_cast<const float4*>(wide + (r + u) * W + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (r + u >= r1) break;
      const bool bias_row = static_cast<int>((r + u) % n_adj) < bias_streams;
      if (kAdjWide && bias_row) { bs[0] += w[u].x; bs[1] += w[u].y; bs[2] += w[u].z; bs[3] += w[u].w; }
#pragma unroll
      for (int j = 0; j < kSkinny; ++j)
        if (j < S) {
          const float v = __ldg(nar + (r + u) * S + j);
          acc[j][0] = fmaf(v, w[u].x, acc[j][0]);
          acc[j][1] = fmaf(v, w[u].y, acc[j][1]);
          acc[j][2] = fmaf(v, w[u].z, acc[j][2]);
          acc[j][3] = fmaf(v, w[u].w, acc[j][3]);
          if (!kAdjWide && bias_row) bn[j] += v;
        }
    }
  }
#pragma unroll
  for (int j = 0; j < kSkinny; ++j)
    if (j < S) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        // dW is (N, K) row-major: wide = adj -> element (n = c + e, k = j); wide = in -> element (n = j, k = c + e)
        const size_t idx = kAdjWide ? static_cast<size_t>(c + e) * K + j : static_cast<size_t>(j) * K + (c + e);
        atomicAdd(&dW[idx], acc[j][e]);
      }
      if (!kAdjWide && c == 0) atomicAdd(&db[j], bn[j]);
    }
  if (kAdjWide) {
#pragma unroll
    for (int e = 0; e < 4; ++e) atomicAdd(&db[c + e], bs[e]);
  }
}

// One "pass" = one net, one batch, one choice of jet streams: transposes, k_jets_fwd, k_jets_bwd, k_wgrad.
struct PassCfg {
  const DmipMlp* net;
  LossProblem prob;            // what the kernels of either family see of the problem
  int has_I, has_T, has_S, has_Q;
  int n_tan;                   // spatial tangent streams (0 = d)
  const float* hutch_v;
  float* grad;
};

// prob.B and the 1 / (global batch) the losses are normalised with (batch_global = 0: this call holds the whole batch)
void set_batch(LossProblem* pb, long long batch, long long batch_global) {
  pb->B = batch;
  pb->inv_B = 1.0f / static_cast<float>(batch_global > 0 ? batch_global : (batch > 0 ? batch : 1));
}

// workspace map of the tcgen05 path (dmip_tcl.cu): packed weight images, stash images, phi'' zd, output adjoints
struct TclPlan {
  bool use;
  TclStreams st;
  long long n_tiles_fwd, n_tiles_bwd;
  size_t off_stages_fwd, off_stages_bwd, off_in[4][2], off_adj[4][2], off_st[3], off_abar, bytes;
};

struct LossPlan {
  int n_streams, spt, n_adj;
  int n_tan;
  size_t off_in[DMIP_MAX_LAYERS], off_adj[DMIP_MAX_LAYERS], off_zdt[DMIP_MAX_LAYERS], off_abar;
  size_t off_tan[DMIP_MAX_LAYERS];
  size_t bytes;
  TclPlan tcl;
};

inline size_t align_1k(size_t v) { return (v + 1023) & ~size_t(1023); }

// The tensor-core path serves [in <= 64] -> 512 -> 512 -> 512 -> [out <= 64] nets (every score net of the reference's
// configs) for the compiled stream sets; everything else — other widths, the grad_x pass of the adjoint Score-FPE route —
// runs the fp32 FFMA kernels of this file.  DMIP_LOSS_PATH=ffma forces the FFMA kernels (A/B measurements, tests).
void plan_tcl(const PassCfg& c, int n_tan, TclPlan* t) {
  const DmipMlp& net = *c.net;
  *t = TclPlan{};
  t->st.has_I = c.has_I; t->st.has_T = c.has_T; t->st.n_tan = n_tan; t->st.has_Q = c.has_Q;
  const char* force = getenv("DMIP_LOSS_PATH");
  const bool shape_ok = net.n_layers == 4 && net.width[0] == 512 && net.width[1] == 512 && net.width[2] == 512 &&
                        net.out_dim <= kTclSmallF && net.in_dim <= kTclSmallF;
  t->use = shape_ok && c.prob.post != 3 && c.prob.B > 0 && tcl_streams_supported(t->st) && !(force && strcmp(force, "ffma") == 0);
  if (!t->use) return;
  const long long B = c.prob.B;
  t->n_tiles_fwd = (B + t->st.spt_fwd() - 1) / t->st.spt_fwd();
  t->n_tiles_bwd = (B + t->st.spt_bwd() - 1) / t->st.spt_bwd();
  const size_t big = static_cast<size_t>(t->n_tiles_bwd) * 512 * 128, small = static_cast<size_t>(t->n_tiles_bwd) * kTclSmallF * 128;
  size_t off = 0;
  t->off_stages_fwd = off; off += align_1k(static_cast<size_t>(kTclFwdStages) * kTclStage);
  t->off_stages_bwd = off; off += align_1k(static_cast<size_t>(kTclBwdStagesIn) * kTclStage);
  for (int l = 0; l < 4; ++l)
    for (int h = 0; h < 2; ++h) {
      t->off_in[l][h] = off;  off += align_1k(l == 0 ? small : big);
      t->off_adj[l][h] = off; off += align_1k(l == 3 ? small : big);
    }
  for (int l = 0; l < 3; ++l) { t->off_st[l] = off; off += align_1k(static_cast<size_t>(B) * t->st.n_adj() * 512 * sizeof(float)); }
  t->off_abar = off; off += align_1k(static_cast<size_t>(B) * t->st.n_adj() * net.out_dim * sizeof(float));
  t->bytes = off;
}

int plan_pass(const PassCfg& c, LossPlan* p) {
  const DmipMlp& net = *c.net;
  const int d = c.prob.d;
  p->n_tan = c.has_S ? (c.n_tan > 0 ? c.n_tan : d) : 0;
  p->n_streams = 1 + c.has_I + c.has_T + p->n_tan + (c.has_Q ? d * (d + 1) / 2 : 0);
  DMIP_REQUIRE(p->n_streams <= kRows, "too many jet streams (%d > %d): the Score-FPE loss with exact divergence supports "
               "d <= %d diffused dimensions; use divergence_method = 'hutchinson' or pde_loss = 'cScoreFPE'",
               p->n_streams, kRows, kRows - 1);
  p->spt = kRows / p->n_streams;
  p->n_adj = 1 + c.has_I + c.has_T;
  const bool gpass = c.prob.post == 3;   // grad_x pass: no adjoint rows / wgrad operands, but the tangents are kept
  size_t off = tile_net_bytes(net);   // the transposed weights lead the workspace (tile_net_stage)
  int k = net.in_dim;
  const size_t B = static_cast<size_t>(c.prob.B);
  for (int l = 0; l < net.n_layers; ++l) {
    const int n = net.width[l];
    p->off_in[l] = off;  off += align_up(sizeof(float) * B * p->n_adj * k);
    p->off_adj[l] = off; off += gpass ? 0 : align_up(sizeof(float) * B * p->n_adj * n);
    p->off_zdt[l] = off; off += (c.has_T && l < net.n_layers - 1) ? align_up(sizeof(float) * B * n) : 0;
    p->off_tan[l] = off; off += (gpass && l < net.n_layers - 1) ? align_up(sizeof(float) * B * p->n_tan * n) : 0;
    k = n;
  }
  p->off_abar = off;
  off += align_up(sizeof(float) * B * (gpass ? 1 + p->n_tan : p->n_adj) * net.out_dim);
  p->bytes = off;
  plan_tcl(c, p->n_tan, &p->tcl);
  if (p->tcl.use) p->bytes = p->tcl.bytes;
  return DMIP_OK;
}

// DmipLoss -> PassCfg (CDE / CDiffE losses), with the reference's argument checks
int cfg_from_loss(const DmipLoss* q, PassCfg* c) {
  DMIP_REQUIRE(q != nullptr, "descriptor is NULL");
  DMIP_REQUIRE(q->kind == DMIP_LOSS_DSM || q->kind == DMIP_LOSS_DSM_PDE || q->kind == DMIP_LOSS_PINN ||
               q->kind == DMIP_LOSS_PINN2,
               "No valid loss_fn was specified. Options are DMIP_LOSS_DSM, DMIP_LOSS_DSM_PDE, DMIP_LOSS_PINN, DMIP_LOSS_PINN2.");
  DMIP_REQUIRE(q->model == DMIP_CDE || q->model == DMIP_CDIFFE, "model must be DMIP_CDE or DMIP_CDIFFE");
  DMIP_REQUIRE(q->xdim >= 1 && q->ydim >= 1 && q->batch >= 0, "xdim/ydim must be positive, batch >= 0");
  int rc = tile_net_check(q->net, q->xdim + q->ydim + 1, "net");
  if (rc) return rc;
  *c = PassCfg{};
  c->net = &q->net;
  LossProblem& pb = c->prob;
  pb.xdim = q->xdim; pb.ydim = q->ydim;
  pb.d = (q->model == DMIP_CDE) ? q->xdim : q->xdim + q->ydim;
  pb.cdim = (q->model == DMIP_CDE) ? q->ydim : 0;
  DMIP_REQUIRE(q->net.out_dim == pb.d, "s and x_t need to have the same shape, but out_dim %d and %d was given",
               q->net.out_dim, pb.d);
  const bool pde = q->kind != DMIP_LOSS_DSM;
  if (pde) {
    DMIP_REQUIRE(q->pde_loss == DMIP_PDE_FPE || q->pde_loss == DMIP_PDE_CFPE, "pde_loss must be FPE or cScoreFPE");
    DMIP_REQUIRE(q->pde_metric == DMIP_L1 || q->pde_metric == DMIP_L2,
                 "No valid metric specified. Metric should be one of \"L1\" or \"L2\"");
  }
  const bool pinn = q->kind == DMIP_LOSS_PINN || q->kind == DMIP_LOSS_PINN2;
  if (pinn) {
    DMIP_REQUIRE(q->ic_metric == DMIP_L1 || q->ic_metric == DMIP_L2, "ic_metric should be one of \"L1\" or \"L2\"");
    DMIP_REQUIRE(q->ic_target != nullptr || q->batch == 0, "PINNLoss needs ic_target = initial_condition(x, y)");
  }
  c->has_I = pinn;
  c->has_T = pde;
  const bool fpe = pde && q->pde_loss == DMIP_PDE_FPE;
  if (fpe) {
    DMIP_REQUIRE(q->divergence == DMIP_DIV_EXACT || q->divergence == DMIP_DIV_HUTCHINSON ||
                 q->divergence == DMIP_DIV_EXACT_ADJOINT,
                 "No valid value for divergence method specified. Need to be one of \"exact\",\"hutchinson\",\"approx\" or "
                 "\"approximate\"");
    DMIP_REQUIRE(q->divergence != DMIP_DIV_HUTCHINSON || q->hutch_v != nullptr || q->batch == 0,
                 "divergence = hutchinson needs the probe vectors hutch_v (batch, d)");
  }
  // forward-only route (second-order streams) for small d, adjoint route (grad_x pass + reverse sweep) otherwise
  pb.gx = fpe && (q->divergence != DMIP_DIV_EXACT || pb.d > kMaxD);
  c->has_S = fpe && !pb.gx;
  c->has_Q = c->has_S;
  pb.kind = q->kind; pb.model = q->model;
  pb.pde_loss = q->pde_loss; pb.pde_metric = q->pde_metric; pb.ic_metric = q->ic_metric;
  set_batch(&pb, q->batch, q->batch_global);
  pb.bmin = q->beta_min; pb.bmax = q->beta_max; pb.lam = q->lam; pb.lam2 = q->lam2;
  pb.x = q->x; pb.y = q->y; pb.t = q->t; pb.eps = q->eps; pb.ic_target = q->ic_target;
  pb.losses = q->out_losses; c->grad = q->grad;
  return DMIP_OK;
}

// dst[j] += sum_r src[r][j]  (few columns: one block per 256-row slab, smem-free warp reductions)
__global__ void __launch_bounds__(256) k_colsum(const float* __restrict__ src, float* dst, long long rows, int cols) {
  for (int j = 0; j < cols; ++j) {
    float acc = 0.f;
    for (long long r = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; r < rows;
         r += static_cast<long long>(gridDim.x) * blockDim.x)
      acc += src[r * cols + j];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if ((threadIdx.x & 31) == 0) atomicAdd(&dst[j], acc);
  }
}

int launch_colsum(const float* src, float* dst, long long rows, int cols, cudaStream_t s) {
  const long long blocks = (rows + 255) / 256;
  k_colsum<<<static_cast<unsigned>(blocks < 592 ? blocks : 592), 256, 0, s>>>(src, dst, rows, cols);
  DMIP_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return DMIP_OK;
}

int g_loss_sm = 0;
bool g_loss_ready[64] = {};   // cudaFuncSetAttribute is per device
constexpr int kLossSmem = (2 * kMaxW * kLd + kWbufFloats) * 4;

int loss_init() {
  int dev = 0;
  DMIP_CHECK_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || !g_loss_ready[dev]) {
    int n = 0;
    DMIP_CHECK_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
    DMIP_CHECK_CUDA(cudaFuncSetAttribute(k_jets_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, kLossSmem));
    DMIP_CHECK_CUDA(cudaFuncSetAttribute(k_jets_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, kLossSmem));
    DMIP_CHECK_CUDA(cudaFuncSetAttribute(k_gradx_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, kLossSmem));
    g_loss_sm = n;
    if (dev >= 0 && dev < 64) g_loss_ready[dev] = true;
  }
  return DMIP_OK;
}

// Device view of a pass on the tcgen05 kernels: the problem, the net, the stream set and the workspace map of the plan.
TclDev tcl_dev(const PassCfg& c, const TclPlan& t, uint8_t* ws) {
  const DmipMlp& net = *c.net;
  TclDev D{c.prob};
  D.stages_fwd = ws + t.off_stages_fwd;
  D.stages_bwd = ws + t.off_stages_bwd;
  long long off = 0;
  int k = net.in_dim;
  for (int l = 0; l < 4; ++l) {
    D.W[l] = net.W[l];
    D.b[l] = net.b[l];
    off += static_cast<long long>(net.width[l]) * k;
    D.off_b[l] = off;
    off += net.width[l];
    k = net.width[l];
    for (int h = 0; h < 2; ++h) {
      D.in_img[l][h] = ws + t.off_in[l][h];
      D.adj_img[l][h] = ws + t.off_adj[l][h];
    }
    if (l < 3) D.st[l] = reinterpret_cast<float*>(ws + t.off_st[l]);
  }
  D.in_dim = net.in_dim; D.out_dim = net.out_dim;
  D.k0steps_fwd = (net.in_dim + 15) / 16;
  D.k0steps_bwd = (net.out_dim + 15) / 16;
  D.has_I = t.st.has_I; D.has_T = t.st.has_T; D.n_tan = t.st.n_tan; D.has_Q = t.st.has_Q;
  D.abar = reinterpret_cast<float*>(ws + t.off_abar);   // post = 4: unused by the forward; the backward takes grad_out
  D.grad = c.grad;
  D.n_tiles_fwd = t.n_tiles_fwd; D.n_tiles_bwd = t.n_tiles_bwd;
  return D;
}

// One pass on the tcgen05 kernels: weight images, forward (loss terms, output adjoints, stashes), backward, four
// weight-gradient GEMMs.
int run_pass_tcl(const PassCfg& c, const LossPlan& p, uint8_t* ws, cudaStream_t s) {
  const DmipMlp& net = *c.net;
  const TclDev D = tcl_dev(c, p.tcl, ws);
  int rc;
  if ((rc = tcl_launch_pack(D, s))) return rc;
  DMIP_CHECK_CUDA(cudaMemsetAsync(c.grad, 0, loss_grad_floats(&net) * sizeof(float), s));
  if ((rc = tcl_launch_fwd(D, s))) return rc;
  if ((rc = tcl_launch_bwd(D, s))) return rc;
  return tcl_launch_wgrad(D, s);
}

// Enqueue one pass.  `ws` must hold p.bytes; c.grad is zeroed here, c.prob.losses is NOT (the caller owns it).
int run_pass(const PassCfg& c, const LossPlan& p, uint8_t* ws, cudaStream_t s) {
  if (p.tcl.use) return run_pass_tcl(c, p, ws, s);
  int rc = loss_init();
  if (rc) return rc;
  const int n_sm = g_loss_sm;
  const DmipMlp& net = *c.net;
  const LossProblem& pb = c.prob;
  LossDev D{pb};
  if ((rc = tile_net_stage(net, ws, &D, s))) return rc;
  D.has_I = c.has_I; D.has_T = c.has_T; D.has_S = c.has_S; D.has_Q = c.has_Q;
  D.n_streams = p.n_streams; D.spt = p.spt; D.n_adj = p.n_adj;
  D.n_tan = p.n_tan; D.hutch_v = c.hutch_v;
  D.abar = reinterpret_cast<float*>(ws + p.off_abar);
  for (int l = 0; l < net.n_layers; ++l) {
    D.W[l] = net.W[l];
    D.in_rows[l] = reinterpret_cast<float*>(ws + p.off_in[l]);
    D.adj_rows[l] = reinterpret_cast<float*>(ws + p.off_adj[l]);
    D.zdt[l] = reinterpret_cast<float*>(ws + p.off_zdt[l]);
    D.tan_z[l] = reinterpret_cast<float*>(ws + p.off_tan[l]);
  }
  if (pb.post != 3) DMIP_CHECK_CUDA(cudaMemsetAsync(c.grad, 0, loss_grad_floats(&net) * sizeof(float), s));
  if (pb.B == 0) return DMIP_OK;

  const long long tiles_f = (pb.B + p.spt - 1) / p.spt;
  k_jets_fwd<<<static_cast<unsigned>(tiles_f < 4LL * n_sm ? tiles_f : 4LL * n_sm), kThreadsL, kLossSmem, s>>>(D);
  DMIP_CHECK_CUDA(cudaGetLastError());
  count_launch();
  if (pb.post == 3) {   // grad_x pass: reverse sweep to the inputs only
    const int spt_g = kRows / (1 + p.n_tan);
    const long long tiles_g = (pb.B + spt_g - 1) / spt_g;
    k_gradx_bwd<<<static_cast<unsigned>(tiles_g < 4LL * n_sm ? tiles_g : 4LL * n_sm), kThreadsL, kLossSmem, s>>>(D);
    DMIP_CHECK_CUDA(cudaGetLastError());
    count_launch();
    return DMIP_OK;
  }
  const int spt_b = kRows / p.n_adj;
  const long long tiles_b = (pb.B + spt_b - 1) / spt_b;
  k_jets_bwd<<<static_cast<unsigned>(tiles_b < 4LL * n_sm ? tiles_b : 4LL * n_sm), kThreadsL, kLossSmem, s>>>(D);
  DMIP_CHECK_CUDA(cudaGetLastError());
  count_launch();

  // weight / bias gradients, flat layout [W_0, b_0, W_1, b_1, ...]
  float* g = c.grad;
  int k = net.in_dim;
  const long long rows = pb.B * p.n_adj;
  for (int l = 0; l < net.n_layers; ++l) {
    const int n = net.width[l];
    if ((k <= kSkinny && n % 4 == 0 && n > kSkinny) || (n <= kSkinny && k % 4 == 0 && k > kSkinny)) {
      const bool adj_wide = k <= kSkinny;
      const int wide = adj_wide ? n : k;
      const int col_blocks = ceil_div(wide, 512);
      long long ctas = 8LL * n_sm / col_blocks;
      if (ctas > (rows + 63) / 64) ctas = (rows + 63) / 64;
      if (ctas < 1) ctas = 1;
      const long long rpc = (rows + ctas - 1) / ctas;
      dim3 grid(static_cast<unsigned>((rows + rpc - 1) / rpc), col_blocks);
      if (adj_wide)
        k_wgrad_skinny<true><<<grid, 128, 0, s>>>(D.adj_rows[l], D.in_rows[l], g, g + static_cast<size_t>(n) * k, rows, n, k,
                                                  p.n_adj, 1 + c.has_I, rpc);
      else
        k_wgrad_skinny<false><<<grid, 128, 0, s>>>(D.adj_rows[l], D.in_rows[l], g, g + static_cast<size_t>(n) * k, rows, n, k,
                                                   p.n_adj, 1 + c.has_I, rpc);
      DMIP_CHECK_CUDA(cudaGetLastError());
      count_launch();
      g += static_cast<size_t>(n) * k + n;
      k = n;
      continue;
    }
    const int tiles = ceil_div(n, kWgT) * ceil_div(k, kWgT);
    int split = (2 * n_sm) / tiles;   // two CTAs are resident per SM: one full wave, never a nearly empty second one
    const long long max_split = (rows + 255) / 256;
    if (split > max_split) split = static_cast<int>(max_split);
    if (split < 1) split = 1;
    long long rps = (rows + split - 1) / split;
    rps = (rps + p.n_adj * kWgR - 1) / (p.n_adj * kWgR) * (p.n_adj * kWgR);   // keep stream phase aligned per split
    split = static_cast<int>((rows + rps - 1) / rps);
    dim3 grid(ceil_div(k, kWgT), ceil_div(n, kWgT), split);
    k_wgrad<<<grid, 256, 0, s>>>(D.adj_rows[l], D.in_rows[l], g, g + static_cast<size_t>(n) * k, rows, n, k, p.n_adj,
                                 1 + c.has_I, rps);
    DMIP_CHECK_CUDA(cudaGetLastError());
    count_launch();
    g += static_cast<size_t>(n) * k + n;
    k = n;
  }
  return DMIP_OK;
}

// target = std^2 J_s^T u + u  (losses.py:369)  — in place over u
__global__ void k_post_target(const float* __restrict__ J, float* __restrict__ u, const float* __restrict__ t, long long B,
                              int d, float bmin, float bmax) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= B) return;
  float beta, alpha, var;
  vp_terms<false>(t[i], bmin, bmax, beta, alpha, var);
  float uu[8], out[8];
  for (int j = 0; j < d; ++j) uu[j] = u[i * d + j];
  for (int k = 0; k < d; ++k) {
    float acc = 0.f;
    for (int j = 0; j < d; ++j) acc = fmaf(J[(i * d + j) * d + k], uu[j], acc);
    out[k] = fmaf(var, acc, uu[k]);
  }
  for (int k = 0; k < d; ++k) u[i * d + k] = out[k];
}

struct PostPlan {
  PassCfg c1, c2;
  LossPlan p1, p2;
  size_t off_pass, off_s, off_J, off_x0, off_xt, off_surr, bytes;
  DmipSurrogate sd;
};

int plan_posterior(const DmipPosteriorLoss* q, PostPlan* P) {
  DMIP_REQUIRE(q != nullptr, "descriptor is NULL");
  DMIP_REQUIRE(q->xdim >= 1 && q->xdim <= kMaxD && q->ydim >= 1 && q->batch >= 0,
               "PosteriorLoss: 1 <= xdim <= %d (Jacobian tangent streams), ydim >= 1", kMaxD);
  int rc;
  if ((rc = tile_net_check(q->prior_net, q->xdim + 1, "prior_net"))) return rc;
  if ((rc = tile_net_check(q->lik_net, q->xdim + q->ydim + 1, "likelihood_net"))) return rc;
  if ((rc = tile_net_check(q->surrogate, q->xdim, "forward_model"))) return rc;
  DMIP_REQUIRE(q->prior_net.out_dim == q->xdim && q->lik_net.out_dim == q->xdim && q->surrogate.out_dim == q->ydim,
               "PosteriorLoss: prior/likelihood nets must output xdim columns and the forward model ydim");
  PassCfg base = {};
  LossProblem& pb = base.prob;
  pb.xdim = q->xdim; pb.ydim = q->ydim; pb.d = q->xdim;
  pb.kind = DMIP_LOSS_DSM; pb.model = DMIP_CDE;
  set_batch(&pb, q->batch, q->batch_global);
  pb.bmin = q->beta_min; pb.bmax = q->beta_max; pb.lam = q->lam;
  pb.x = q->x; pb.y = q->y; pb.t = q->t; pb.eps = q->eps;
  pb.losses = q->out_losses;
  P->c1 = base;
  P->c1.net = &q->prior_net; P->c1.prob.cdim = 0; P->c1.has_S = 1; P->c1.prob.post = 1; P->c1.grad = q->grad_prior;
  P->c2 = base;
  P->c2.net = &q->lik_net; P->c2.prob.cdim = q->ydim; P->c2.prob.post = 2; P->c2.grad = q->grad_lik;
  if ((rc = plan_pass(P->c1, &P->p1))) return rc;
  if ((rc = plan_pass(P->c2, &P->p2))) return rc;
  const size_t B = static_cast<size_t>(q->batch), d = q->xdim;
  size_t off = 0;
  P->off_pass = off; off += P->p1.bytes > P->p2.bytes ? P->p1.bytes : P->p2.bytes;   // the passes run one after the other
  P->off_s = off;  off += align_up(sizeof(float) * B * d);
  P->off_J = off;  off += align_up(sizeof(float) * B * d * d);
  P->off_x0 = off; off += align_up(sizeof(float) * B * d);
  P->off_xt = off; off += align_up(sizeof(float) * B * d);
  P->sd = DmipSurrogate{};
  P->sd.mode = DMIP_SURR_LIK_VJP;
  P->sd.net = q->surrogate;
  P->sd.a = q->a; P->sd.b = q->b; P->sd.lambd_bd = 0.f;
  P->sd.n = q->batch;
  P->off_surr = off; off += surrogate_workspace(&P->sd);
  P->bytes = off;
  return DMIP_OK;
}

}  // namespace

namespace {

// main pass, preceded by the grad_x pass when the Score-FPE term takes the adjoint route
struct FullPlan {
  PassCfg c, cg;
  LossPlan p, pg;
  bool two;
  size_t off_gradx, bytes;
};

int plan_loss(const DmipLoss* q, FullPlan* F) {
  int rc = cfg_from_loss(q, &F->c);
  if (rc) return rc;
  if ((rc = plan_pass(F->c, &F->p))) return rc;
  F->two = F->c.prob.gx != 0;
  F->off_gradx = 0;
  F->bytes = F->p.bytes;
  if (F->two) {
    F->cg = F->c;
    F->cg.has_I = 0; F->cg.has_T = 0; F->cg.has_S = 1; F->cg.has_Q = 0; F->cg.prob.gx = 0; F->cg.prob.post = 3;
    F->cg.prob.kind = DMIP_LOSS_DSM;
    F->cg.n_tan = (q->divergence == DMIP_DIV_HUTCHINSON) ? 1 : F->c.prob.d;
    F->cg.hutch_v = (q->divergence == DMIP_DIV_HUTCHINSON) ? q->hutch_v : nullptr;
    if ((rc = plan_pass(F->cg, &F->pg))) return rc;
    const size_t pass = F->p.bytes > F->pg.bytes ? F->p.bytes : F->pg.bytes;   // the passes run one after the other
    F->off_gradx = pass;
    F->bytes = pass + align_up(sizeof(float) * static_cast<size_t>(q->batch) * F->c.prob.d);
  }
  return DMIP_OK;
}

}  // namespace

size_t loss_workspace(const DmipLoss* q) {
  FullPlan F;
  if (plan_loss(q, &F)) return 0;
  return F.bytes > 16 ? F.bytes : 16;
}

size_t loss_grad_floats(const DmipMlp* net) {
  size_t n = 0;
  int k = net->in_dim;
  for (int l = 0; l < net->n_layers; ++l) {
    n += static_cast<size_t>(k) * net->width[l] + net->width[l];
    k = net->width[l];
  }
  return n;
}

int launch_loss(const DmipLoss* q, cudaStream_t s) {
  FullPlan F;
  int rc = plan_loss(q, &F);
  if (rc) return rc;
  DMIP_REQUIRE(q->out_losses && q->grad, "out_losses / grad is NULL");
  DMIP_REQUIRE(q->batch == 0 || (q->x && q->y && q->t && q->eps), "x / y / t / eps is NULL");
  if (!q->workspace || q->workspace_bytes < F.bytes || (reinterpret_cast<uintptr_t>(q->workspace) & 15)) {
    set_error("workspace too small or misaligned: need %zu bytes", F.bytes);
    return DMIP_EWORKSPACE;
  }
  uint8_t* ws = static_cast<uint8_t*>(q->workspace);
  DMIP_CHECK_CUDA(cudaMemsetAsync(q->out_losses, 0, 4 * sizeof(float), s));
  if (F.two) {
    float* gradx = reinterpret_cast<float*>(ws + F.off_gradx);
    F.cg.prob.gradx = gradx;
    F.c.prob.gradx = gradx;
    if ((rc = run_pass(F.cg, F.pg, ws, s))) return rc;
  }
  return run_pass(F.c, F.p, ws, s);
}

// ------------------------------------------------------------------------------------------------ plain net forward / backward
namespace {

int mlp_grad_plan(const DmipMlpGrad* q, PassCfg* c, LossPlan* p) {
  DMIP_REQUIRE(q != nullptr && q->n >= 0, "descriptor is NULL or n < 0");
  DMIP_REQUIRE(q->x_dim >= 1 && q->cond_dim >= 0 && q->x_dim + q->cond_dim + 1 == q->net.in_dim,
               "Input Tensor is expected to be 2D with x_dim+cond_dim+1 = %d columns (net.in_dim = %d)",
               q->x_dim + q->cond_dim + 1, q->net.in_dim);
  int rc = tile_net_check(q->net, q->net.in_dim, "net");
  if (rc) return rc;
  *c = PassCfg{};
  c->net = &q->net;
  LossProblem& pb = c->prob;
  pb.xdim = q->x_dim; pb.ydim = q->cond_dim; pb.d = q->x_dim; pb.cdim = q->cond_dim;
  pb.post = 4;
  pb.kind = DMIP_LOSS_DSM; pb.model = DMIP_CDE;
  set_batch(&pb, q->n, q->n);   // post = 4 has no loss stage: inv_B only scales the zero loss sums into scratch
  pb.x = q->x; pb.y = q->cond; pb.t = q->t;
  if ((rc = plan_pass(*c, p))) return rc;
  DMIP_REQUIRE(p->tcl.use || q->n == 0, "dmip_mlp_forward_stash serves [in <= 64] -> 512 -> 512 -> 512 -> [out <= 64] nets "
               "(tcgen05 kernels); use the module's own autograd for other shapes");
  return DMIP_OK;
}

int mlp_grad_check_ws(const DmipMlpGrad* q, const LossPlan& p) {
  if (!q->workspace || q->workspace_bytes < p.bytes || (reinterpret_cast<uintptr_t>(q->workspace) & 1023)) {
    set_error("workspace too small or not 1024-byte aligned: need %zu bytes", p.bytes);
    return DMIP_EWORKSPACE;
  }
  return DMIP_OK;
}

}  // namespace

size_t mlp_grad_workspace(const DmipMlpGrad* q) {
  PassCfg c;
  LossPlan p;
  if (mlp_grad_plan(q, &c, &p) || !p.tcl.use) return 0;
  return p.bytes;
}

int launch_mlp_forward_stash(const DmipMlpGrad* q, cudaStream_t s) {
  PassCfg c;
  LossPlan p;
  int rc = mlp_grad_plan(q, &c, &p);
  if (rc) return rc;
  if (q->n == 0) return DMIP_OK;
  DMIP_REQUIRE(q->x && q->t && q->out && (q->cond || q->cond_dim == 0), "x / cond / t / out is NULL");
  if ((rc = mlp_grad_check_ws(q, p))) return rc;
  TclDev D = tcl_dev(c, p.tcl, static_cast<uint8_t*>(q->workspace));
  D.net_out = q->out;
  // the forward never touches grad / losses in this mode, but its epilogue addresses them unconditionally at the end:
  // point them at scratch inside the (not yet used) adjoint image of the output layer
  D.grad = reinterpret_cast<float*>(D.adj_img[0][0]);
  D.losses = reinterpret_cast<float*>(D.adj_img[0][1]);
  for (int l = 0; l < 4; ++l) D.off_b[l] = 0;
  if ((rc = tcl_launch_pack(D, s))) return rc;      // both images: the backward must see the weights of THIS forward
  return tcl_launch_fwd(D, s);
}

int launch_mlp_backward(const DmipMlpGrad* q, cudaStream_t s) {
  PassCfg c;
  LossPlan p;
  int rc = mlp_grad_plan(q, &c, &p);
  if (rc) return rc;
  DMIP_REQUIRE(q->grad_params != nullptr, "grad_params is NULL");
  DMIP_CHECK_CUDA(cudaMemsetAsync(q->grad_params, 0, loss_grad_floats(&q->net) * sizeof(float), s));
  if (q->n == 0) return DMIP_OK;
  DMIP_REQUIRE(q->grad_out != nullptr, "grad_out is NULL");
  if ((rc = mlp_grad_check_ws(q, p))) return rc;
  TclDev D = tcl_dev(c, p.tcl, static_cast<uint8_t*>(q->workspace));
  D.abar = const_cast<float*>(q->grad_out);
  D.grad = q->grad_params;
  D.grad_in = q->grad_in;
  if ((rc = tcl_launch_bwd(D, s))) return rc;
  if ((rc = tcl_launch_wgrad(D, s))) return rc;
  // d / d b_3 = column sums of grad_out (the loss kernels get it from their own loss stage): one small reduction
  return launch_colsum(q->grad_out, q->grad_params + (loss_grad_floats(&q->net) - q->net.out_dim), q->n, q->net.out_dim, s);
}

size_t posterior_loss_workspace(const DmipPosteriorLoss* q) {
  PostPlan P;
  if (plan_posterior(q, &P)) return 0;
  return P.bytes;
}

int launch_posterior_loss(const DmipPosteriorLoss* q, cudaStream_t s) {
  PostPlan P;
  int rc = plan_posterior(q, &P);
  if (rc) return rc;
  DMIP_REQUIRE(q->out_losses && q->grad_prior && q->grad_lik, "out_losses / grad_prior / grad_lik is NULL");
  DMIP_REQUIRE(q->batch == 0 || (q->x && q->y && q->t && q->eps), "x / y / t / eps is NULL");
  if (!q->workspace || q->workspace_bytes < P.bytes || (reinterpret_cast<uintptr_t>(q->workspace) & 15)) {
    set_error("workspace too small or misaligned: need %zu bytes", P.bytes);
    return DMIP_EWORKSPACE;
  }
  uint8_t* ws = static_cast<uint8_t*>(q->workspace);
  float* aux_s = reinterpret_cast<float*>(ws + P.off_s);
  float* aux_J = reinterpret_cast<float*>(ws + P.off_J);
  float* aux_x0 = reinterpret_cast<float*>(ws + P.off_x0);
  float* aux_xt = reinterpret_cast<float*>(ws + P.off_xt);
  DMIP_CHECK_CUDA(cudaMemsetAsync(q->out_losses, 0, 4 * sizeof(float), s));
  // 1. prior net: DSM + its gradient; s_prior, J_s, Tweedie mean x0_hat
  P.c1.prob.aux_s = aux_s; P.c1.prob.aux_J = aux_J; P.c1.prob.aux_x0 = aux_x0; P.c1.prob.aux_xt = aux_xt;
  if ((rc = run_pass(P.c1, P.p1, ws + P.off_pass, s))) return rc;
  if (q->batch > 0) {
    // 2. u = J_f(x0_hat)^T (-a^2 v1 + v2 + a^2 v3)  -> aux_s
    P.sd.x = aux_x0; P.sd.y = q->y; P.sd.grad = aux_s;
    P.sd.workspace = ws + P.off_surr; P.sd.workspace_bytes = surrogate_workspace(&P.sd);
    if ((rc = launch_surrogate(&P.sd, s))) return rc;
    // 3. target = std^2 J_s^T u + u
    k_post_target<<<static_cast<unsigned>((q->batch + 255) / 256), 256, 0, s>>>(aux_J, aux_s, q->t, q->batch, q->xdim,
                                                                                 q->beta_min, q->beta_max);
    DMIP_CHECK_CUDA(cudaGetLastError());
    count_launch();
  }
  // 4. likelihood net: lam * sum (alpha s_lik - target)^2 + its gradient
  P.c2.prob.aux_s = aux_s;
  return run_pass(P.c2, P.p2, ws + P.off_pass, s);
}

}  // namespace dmip
