// dmip_jets.cuh — the per-sample jet and loss arithmetic of the fused score-training losses, shared by the fp32 FFMA
// kernels (dmip_loss.cu) and the tcgen05 kernels (dmip_tcl.cu).
//
// A sample's streams (dmip_loss.cu header) sit in the order  P | I? | T? | S_0..S_{n_tan-1}? | Q_(i,k), i<=k ?.  The
// functions here take that layout as a template parameter S with the members kI, kT (stream present), sI, sT, sS, sQ
// (stream offsets) and NADJ (adjoint streams P [, I] [, T]): dmip_tcl.cu's Cfg has them as compile-time constants,
// dmip_loss.cu fills the same names at run time.
//
// The SDE (P.sde_kind, uniform per launch) enters through the per-sample terms of sample_sde and a few branches below;
// the VP arithmetic is the same, operation for operation, as before the VE-SDE was added.  With s = a / g:
//   VP:  g^2 = beta, alpha = exp(-B / 2), var = 1 - exp(-B),  d ln g / dt = beta' / (2 beta),
//        Score-FPE  ds/dt = beta / 2 grad_x [div s + |s|^2 + x.s]
//   VE:  g^2 = 2 lr sigma^2, alpha = 1, var = sigma^2,  d ln g / dt = lr = ln(smax / smin),  dz_t/dt = eps sigma lr,
//        Score-FPE  ds/dt = g^2 / 2 grad_x [div s + |s|^2]   (f = 0: no x.s term)
#pragma once
#include "dmip_common.h"
#include "dmip_sde.cuh"

namespace dmip {

// offset of Q_(i,k), i <= k, after the first second-order stream
__device__ __forceinline__ int q_index(int i, int k, int d) { return i * d - (i * (i - 1)) / 2 + (k - i); }

// clean state component k < d of sample smp: CDE: z0 = x; CDiffE: z0 = [x, y]   (models/diffusion.py:80,129)
__device__ __forceinline__ float state0(const LossProblem& P, long long smp, int k) {
  return (k < P.xdim) ? P.x[smp * P.xdim + k] : P.y[smp * P.ydim + (k - P.xdim)];
}

// SDE terms of a sample at its time t: beta = g^2 (VP: beta(t)), alpha, var, sd = sqrt(var); lr (VE only) = ln(smax / smin)
struct SampleSde {
  float t, beta, alpha, var, sd, lr;
};
__device__ __forceinline__ SampleSde sample_sde(const LossProblem& P, long long smp) {
  SampleSde v;
  v.t = P.t[smp];
  if (P.sde_kind == kSdeVE) {
    ve_terms<false>(v.t, P.bmin, P.bmax, v.beta, v.var, v.lr);
    v.alpha = 1.f;
  } else {
    vp_terms<false>(v.t, P.bmin, P.bmax, v.beta, v.alpha, v.var);
    v.lr = 0.f;
  }
  v.sd = sqrtf(v.var);
  return v;
}

// Layer-0 input column k of stream st of sample smp.
template <class S>
__device__ __forceinline__ float jet_input(const LossProblem& P, const S& s, const SampleSde& vp, long long smp, int st,
                                           int k) {
  const int d = P.d;
  float z0k = 0.f, epsk = 0.f;
  if (k < d) {
    z0k = state0(P, smp, k);
    epsk = P.eps[smp * d + k];
  }
  if (st == 0) {                                   // P: [z_t, cond, t]           (sdes.py:43-46)
    if (k < d) return epsk * vp.sd + vp.alpha * z0k;
    if (k < d + P.cdim) return P.y[smp * P.ydim + (k - d)];
    return vp.t;
  }
  if (s.kI && st == s.sI) {                        // I: [x, y, 0]                (losses.py:221-223)
    if (k < P.xdim) return P.x[smp * P.xdim + k];
    if (k < P.xdim + P.ydim) return P.y[smp * P.ydim + (k - P.xdim)];
    return 0.f;
  }
  if (s.kT && st == s.sT) {                        // T: (dz_t/dt, 0, 1)          (SURVEY.md Q8 / App. A.4)
    if (k < d) {
      if (P.sde_kind == kSdeVE) return epsk * vp.sd * vp.lr;
      return epsk * vp.beta * (1.f - vp.var) / (2.f * vp.sd) - 0.5f * vp.beta * vp.alpha * z0k;
    }
    return (k < d + P.cdim) ? 0.f : 1.f;
  }
  return (st >= s.sS && st < s.sQ && k == st - s.sS) ? 1.f : 0.f;   // S_k: e_k;   Q: zero input
}

// Loss terms of output component j of sample smp (set in l_dsm, l_ic, l_pde for the terms the pass has; the caller
// zeroes them) and the adjoints of the net outputs, abar[(smp * NADJ + a) * od + j] for the adjoint streams a = P | I | T.
// o.primal(s, c) is output c of the primal stream s (P or I) with the output bias, o.tangent(s, c) that of a tangent
// stream (T, S_k, Q).  Returns d loss / d b_out[j].
template <class S, class O>
__device__ __forceinline__ float jet_loss_item(const LossProblem& P, const S& s, const O& o, float* abar, int od,
                                               long long smp, int j, float& l_dsm, float& l_ic, float& l_pde) {
  const int d = P.d;
  const float db = P.bmax - P.bmin;
  const bool ve = P.sde_kind == kSdeVE;
  const SampleSde vp = sample_sde(P, smp);
  const float beta = vp.beta, alpha = vp.alpha, var = vp.var, sd = vp.sd, sb = sqrtf(beta);
  const float aj = o.primal(0, j);
  const float epsj = P.eps[smp * d + j];
  float abP, abI = 0.f;                    // adjoints of the primal outputs j of P and I
  if (P.post == 1) {
    // DPS prior net: s_prior = prior_net(x_t, t) IS the score (no 1/g); DSM on it; Tweedie mean and Jacobian
    // for the likelihood target                                                   (losses.py:374-381)
    const float xt = epsj * sd + alpha * P.x[smp * P.xdim + j];
    const float r = aj * sd + epsj;
    l_dsm = 0.5f * r * r;
    abP = P.inv_B * r * sd;
    P.aux_s[smp * d + j] = aj;
    P.aux_xt[smp * d + j] = xt;
    P.aux_x0[smp * d + j] = (xt + var * aj) / alpha;
    for (int k = 0; k < d; ++k) P.aux_J[(smp * d + j) * d + k] = o.tangent(s.sS + k, j);
  } else if (P.post == 2) {
    // DPS likelihood net: sum_j (alpha s_lik - target)^2, target detached           (losses.py:382)
    const float r = alpha * aj - P.aux_s[smp * d + j];
    l_ic = P.lam * r * r;
    abP = P.inv_B * P.lam * 2.f * r * alpha;
  } else {
    // DSM: 1/2 sum (s std + eps)^2, s = a / g                                      (losses.py:49-52, Q3);
    // PINNLoss2 only reports it ('DSM_eval', losses.py:291): no adjoint
    const float r = aj / sb * sd + epsj;
    l_dsm = 0.5f * r * r;
    abP = P.kind == DMIP_LOSS_PINN2 ? 0.f : P.inv_B * r * sd / sb;
  }
  if (s.kI) {                              // initial condition at t = 0          (losses.py:221-230)
    float g0;                              // g(0): VP sqrt(beta_min), VE smin sqrt(2 lr)
    if (ve) {
      float g2, v0, lr0;
      ve_terms<false>(0.f, P.bmin, P.bmax, g2, v0, lr0);
      g0 = sqrtf(g2);
    } else {
      g0 = sqrtf(P.bmin);
    }
    float g = 0.f;
    if (j < P.xdim) {
      const float diff = o.primal(s.sI, j) / g0 - P.ic_target[smp * P.xdim + j];
      if (P.ic_metric == 2) { l_ic = diff * diff; g = 2.f * diff; }
      else { l_ic = fabsf(diff); g = (diff > 0.f) - (diff < 0.f); }
      l_ic *= P.lam2 / P.xdim;
      g *= P.lam2 / (P.xdim * g0);
    }
    abI = P.inv_B * g;
    abar[(smp * s.NADJ + 1) * od + j] = abI;
  }
  if (s.kT) {
    const float ds_dt = ve ? (o.tangent(s.sT, j) - aj * vp.lr) / sb : o.tangent(s.sT, j) / sb - aj * db / (2.f * beta * sb);
    float g;                               // d loss / d ds_dt[j]
    if (P.pde_loss == 0) {
      // Score-FPE residual R = ds/dt - g^2/2 grad_x[div s + |s|^2 (+ x.s: VP)], grad_x constant (losses.py:88-95, Q9)
      float grad_x;
      if (P.gx) {
        grad_x = P.gradx[smp * d + j];     // adjoint route (k_gradx_bwd), any d
      } else {
        float JTa = 0.f, JTx = 0.f, gtr = 0.f;
        for (int i = 0; i < d; ++i) {
          const float ai = o.primal(0, i);
          const float zti = P.eps[smp * d + i] * sd + alpha * state0(P, smp, i);
          const float Jij = o.tangent(s.sS + j, i);                                  // d a_i / d x_j
          JTa = fmaf(Jij, ai, JTa);
          JTx = fmaf(Jij, zti, JTx);
          gtr += o.tangent(s.sQ + q_index(min(i, j), max(i, j), d), i);            // d^2 a_i / dx_i dx_j
        }
        grad_x = ve ? gtr / sb + 2.f * JTa / beta : gtr / sb + 2.f * JTa / beta + (aj + JTx) / sb;
      }
      const float R = ds_dt - 0.5f * beta * grad_x;
      if (P.pde_metric == 1) { l_pde = fabsf(R); g = (R > 0.f) - (R < 0.f); }
      else { l_pde = R * R; g = 2.f * R; }
      l_pde *= P.lam / d;
      g *= P.lam / d * P.inv_B;
    } else {
      // cScoreFPE: sum_j (std^3 ds/dt - eps g^2 alpha^2 / 2)^2  (VE: alpha = 1)   (losses.py:116-124)
      const float r = sd * sd * sd * ds_dt - 0.5f * epsj * beta * alpha * alpha;
      if (P.pde_metric == 2) { l_pde = r * r; g = 2.f * r; }
      else { l_pde = fabsf(r); g = (r > 0.f) - (r < 0.f); }
      l_pde *= P.lam;
      g *= P.lam * sd * sd * sd * P.inv_B;
    }
    abar[(smp * s.NADJ + 1 + s.kI) * od + j] = g / sb;
    abP += ve ? -g * vp.lr / sb : -g * db / (2.f * beta * sb);
  }
  abar[(smp * s.NADJ + 0) * od + j] = abP;
  return abP + abI;
}

}  // namespace dmip
