// dmip_sde.cuh — closed forms of the forward SDEs and the per-sub-step coefficients of the reverse-time integrators,
// shared by the tcgen05 sampler (dmip_tc.cu) and the fp32 sampler (dmip_f32.cu); the loss kernels take vp_terms and
// ve_terms (dmip_jets.cuh).
//
//   VP  (sdes.py:9-57, the only SDE upstream):  beta(t) = bmin + (bmax - bmin) t,  f = -beta x / 2,  g = sqrt(beta),
//        x_t | x_0 ~ N(alpha x_0, var),  alpha = exp(-B / 2),  var = 1 - exp(-B),  B = int_0^t beta.
//   VE  (Song et al. 2021, eq. 30-31; NOT in the reference — BASELINE.json names it, parity unpinned, SURVEY.md §8f N4):
//        sigma(t) = smin (smax / smin)^t,  f = 0,  g = sigma sqrt(2 ln(smax / smin)),  x_t | x_0 ~ N(x_0, sigma(t)^2).
//
// One sampling step = one PREDICTOR sub-step (Euler–Maruyama on the reverse SDE with the plug-in drift a = g * score,
// sdes.py:77-87) followed by n_corr CORRECTOR sub-steps (Langevin dynamics at the new time level: x += e s + sqrt(2 e) z,
// Song et al. 2021 Alg. 4/5).  The Langevin step size is the closed form of Song's norm rule for a calibrated score,
// e = 2 snr^2 std(t)^2  (|z| ~ sqrt(d), |s| ~ sqrt(d) / std): it needs no reduction over a particle's coordinates or
// over the batch, so particles stay independent and the kernel persistent.  Every sub-step has the form
//        x <- x (1 + kx) + ke * eps + ca * net,      net = a  (CDE / CDiffE)   or   prior + likelihood  (DPS, a = g * net)
// at time tau; sub-step u is also the Philox "step" key and the row index of injected noise.
#pragma once
#include <cuda_runtime.h>

namespace dmip {

constexpr int kSdeVP = 0;
constexpr int kSdeVE = 1;

struct SdeSched {
  int kind;          // kSdeVP / kSdeVE
  int S;             // sampling steps
  int n_corr;        // corrector sub-steps per step
  float T;
  float p0, p1;      // VP: beta_min, beta_max;  VE: sigma_min, sigma_max
  float snr;         // corrector signal-to-noise ratio (Song: 0.16)
  float delta, sqrt_delta;   // T / S and its root (models/diffusion.py:31)
};

struct SdeCoef {
  float tau, kx, ke, ca;
  float g, fx;       // predictor sub-steps: g(tau) and the drift factor (-f = fx * x); the fp32 kernel evaluates the
  int corrector;     // reference's own expression  x + delta (g a + fx x) + sqrt(delta) g eps  with them
};

__host__ __device__ inline int sde_substeps(const SdeSched& s) { return s.S * (1 + s.n_corr); }

// time level of sub-step u
__device__ __forceinline__ float sde_tau(int i, int S, float T);
__device__ __forceinline__ float sde_substep_tau(const SdeSched& s, int u) {
  const int per = 1 + s.n_corr;
  const int i = u / per;
  return sde_tau(u - i * per == 0 ? i : i + 1, s.S, s.T);
}

// T - linspace(0, 1, S + 1)[i] * T in fp32, linspace evaluated symmetrically as torch does (models/diffusion.py:34)
__device__ __forceinline__ float sde_tau(int i, int S, float T) {
  const float step = 1.0f / static_cast<float>(S);
  const int steps = S + 1;
  const float l = (i < steps / 2) ? step * static_cast<float>(i) : 1.0f - step * static_cast<float>(steps - i - 1);
  return T - l * T;
}

// VP closed forms at time t (sdes.py:9-49): beta(t) and the moments of x_t | x_0, mean weight alpha and variance var.
// kFast: the intrinsic exp of the tcgen05 sampler (as its VP code always used); the fp32 sampler and the loss kernels
// take the accurate function.
template <bool kFast>
__device__ __forceinline__ void vp_terms(float t, float bmin, float bmax, float& beta, float& alpha, float& var) {
  const float db = bmax - bmin;
  beta = bmin + db * t;
  const float Bt = 0.5f * t * t * db + t * bmin;
  alpha = kFast ? __expf(-0.5f * Bt) : expf(-0.5f * Bt);
  var = 1.0f - (kFast ? __expf(-Bt) : expf(-Bt));
}

// VE closed forms at time t: g(t)^2 = 2 lr sigma^2, the variance sigma(t)^2 of x_t | x_0 (mean weight 1) and
// lr = ln(smax / smin) = d ln sigma / dt.  kFast as in vp_terms.
template <bool kFast>
__device__ __forceinline__ void ve_terms(float t, float smin, float smax, float& g2, float& var, float& lr) {
  lr = kFast ? __logf(smax / smin) : logf(smax / smin);
  const float sig = smin * (kFast ? __expf(t * lr) : expf(t * lr));
  g2 = sig * sig * 2.0f * lr;
  var = sig * sig;
}

// diffusion coefficient g(t)^2 and the moments of x_t | x_0: mean weight alpha, variance var.  kFast: the intrinsic
// exp / log of the tcgen05 path (as its VP code always used); the fp32 path takes the accurate functions.
template <bool kFast>
__device__ __forceinline__ void sde_terms(const SdeSched& s, float t, float& g2, float& alpha, float& var) {
  if (s.kind == kSdeVE) {
    float lr;
    ve_terms<kFast>(t, s.p0, s.p1, g2, var, lr);
    alpha = 1.0f;
  } else {
    vp_terms<kFast>(t, s.p0, s.p1, g2, alpha, var);
  }
}

// coefficients of sub-step u (dps: the net output is the score sum, not g * score)
template <bool kFast>
__device__ __forceinline__ SdeCoef sde_coef(const SdeSched& s, int u, bool dps) {
  const int per = 1 + s.n_corr;
  const int i = u / per, c = u - i * per;
  SdeCoef k;
  float g2, alpha, var;
  if (c == 0) {                          // predictor: x += delta (g a - f) + sqrt(delta) g eps     (sdes.py:77-87)
    k.tau = sde_tau(i, s.S, s.T);
    sde_terms<kFast>(s, k.tau, g2, alpha, var);
    const float g = sqrtf(g2);
    k.corrector = 0;
    k.g = g;
    k.fx = s.kind == kSdeVE ? 0.0f : 0.5f * g2;                // -f = beta x / 2 for VP, 0 for VE
    k.kx = s.delta * k.fx;
    k.ke = s.sqrt_delta * g;
    k.ca = s.delta * (dps ? g2 : g);
  } else {                               // corrector at the time level the predictor just reached
    k.tau = sde_tau(i + 1, s.S, s.T);
    sde_terms<kFast>(s, k.tau, g2, alpha, var);
    const float e = 2.0f * s.snr * s.snr * var;
    k.corrector = 1;
    k.g = sqrtf(g2);
    k.fx = 0.0f;
    k.kx = 0.0f;
    k.ke = sqrtf(2.0f * e);
    k.ca = dps ? e : e * rsqrtf(g2);                           // score = a / g
  }
  return k;
}

}  // namespace dmip
