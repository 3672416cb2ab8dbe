// dmip_common.h — host-side helpers and descriptors shared by the translation units of libdmip_sm100.so
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/dmip.h"

namespace dmip {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);
void reset_launch_count();

#define DMIP_CHECK_CUDA(expr)                                                              \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      ::dmip::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return DMIP_ECUDA;                                                                   \
    }                                                                                      \
  } while (0)

#define DMIP_REQUIRE(cond, ...)         \
  do {                                  \
    if (!(cond)) {                      \
      ::dmip::set_error(__VA_ARGS__);   \
      return DMIP_EINVAL;               \
    }                                   \
  } while (0)

inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
inline int round_up(int a, int b) { return ceil_div(a, b) * b; }

// Geometry of the packed image of one [in]->512->512->512->[out] net for the tcgen05 path.
struct TcNetGeom {
  int n_varying;   // dv: leading input columns that enter the layer-0 GEMM
  int split;       // layer-0 operand parts (1,2,3); l0_split = 4 (one part, f16 operands) is stored as split = 1, l0_f16 = 1
  int l0_f16;      // layer 0 multiplies f16 x f16 (11 mantissa bits of the state for the MMA count of plain bf16)
  int dvp;         // part stride of the split operand: round_up(dv, 8)
  int k0;          // (split - 1) * dvp + dv
  int k0pad;       // k0 rounded up to 16
  int kb0;         // K-blocks (64) of layer 0
  int out_rows;    // leading output rows kept
  int outpad;      // out_rows rounded up to 16
  int n_stages;    // 16 KB weight stages per net pass: 4*kb0 + 32 + 32 + 8
  size_t stage_bytes() const { return size_t(n_stages) * 16384; }
  // fp32 tail after the stages: b0[512] b1[512] b2[512] b3[128] W0const[512 x n_const] (row-constant input columns)
  int n_const;     // in_dim - dv
  size_t tail_floats() const { return 512 * 3 + 128 + size_t(512) * n_const; }
  size_t bytes() const { return stage_bytes() + tail_floats() * 4; }
};
int tc_net_geom(const DmipMlp* net, int n_varying, int out_rows, int split, TcNetGeom* g);

int device_is_sm100();

// The problem of one loss pass.  The device structs of both kernel families (LossDev in dmip_loss.cu, TclDev in
// dmip_tcl.h) derive from it and add their net and workspace pointers.
struct LossProblem {
  int kind, model, xdim, ydim, d, cdim;
  int post;                           // 0: CDE/CDiffE losses; 1: DPS prior net pass; 2: DPS likelihood net pass;
                                      // 3: grad_x pass of the adjoint Score-FPE route (FFMA: streams P | S_k, no loss);
                                      // 4: plain net forward / backward (tcgen05 only: dmip_mlp_forward_stash / _backward);
                                      // 5: double backward of the plain net (tcgen05 only, streams P | T: dmip_mlp_double_backward)
  int pde_loss, pde_metric, ic_metric;
  int gx;                             // 1: Score-FPE grad_x is read from `gradx` (adjoint route) instead of the Q streams
  long long B;
  float inv_B;                        // 1 / global batch
  int sde_kind;                       // kSdeVP / kSdeVE (dmip_sde.cuh), uniform per launch
  float bmin, bmax, lam, lam2;        // bmin / bmax: beta range (VP) or sigma range (VE), as SdeSched's p0 / p1
  const float *x, *y, *t, *eps, *ic_target;
  float* gradx;                       // post=3 out / gx=1 in: grad_x [div s + |s|^2 + x.s]  (B,d)
  float* aux_s;                       // post=1 out: s_prior (B,d);  post=2 in: target (B,d)
  float* aux_J;                       // post=1 out: J_s (B,d,d) row-major [i][k] = d s_i / d x_k
  float* aux_x0;                      // post=1 out: Tweedie mean x0_hat (B,d)
  float* aux_xt;                      // post=1 out: x_t (B,d)
  float* losses;                      // [4] total, dsm, ic, pde
};

// implemented in the kernel translation units
int launch_pack(const DmipMlp* net, const TcNetGeom& g, void* packed, cudaStream_t s);
int launch_sampler_tc(const DmipSampler* d, cudaStream_t s);
int launch_forward_tc(const DmipForward* d, cudaStream_t s);
int launch_sampler_f32(const DmipSampler* d, cudaStream_t s);
int launch_forward_f32(const DmipForward* d, cudaStream_t s);
size_t sampler_f32_workspace(const DmipSampler* d);
size_t forward_f32_workspace(const DmipForward* d);
size_t loss_workspace(const DmipLoss* q);
size_t loss_grad_floats(const DmipMlp* net);
int launch_loss(const DmipLoss* q, cudaStream_t s);
size_t mlp_grad_workspace(const DmipMlpGrad* q);
int launch_mlp_forward_stash(const DmipMlpGrad* q, cudaStream_t s);
int launch_mlp_backward(const DmipMlpGrad* q, cudaStream_t s);
size_t mlp_double_backward_workspace(const DmipMlpGradGrad* q);
int launch_mlp_double_backward(const DmipMlpGradGrad* q, cudaStream_t s);
size_t posterior_loss_workspace(const DmipPosteriorLoss* q);
int launch_posterior_loss(const DmipPosteriorLoss* q, cudaStream_t s);
int launch_histogramdd(const DmipHistogram* d, cudaStream_t s);
int launch_hist_kl(const void* hp, const void* hq, long long m, double epsilon, double* out, cudaStream_t s);
size_t mmd_workspace(const DmipMmd* d);
int launch_mmd(const DmipMmd* d, cudaStream_t s);
size_t mmd_test_workspace(const DmipMmdTest* d);
int launch_mmd_test(const DmipMmdTest* d, cudaStream_t s);
size_t ksd_workspace(const DmipKsd* d);
int launch_ksd(const DmipKsd* d, cudaStream_t s);
size_t surrogate_workspace(const DmipSurrogate* d);
int launch_surrogate(const DmipSurrogate* d, cudaStream_t s);
bool surrogate_tc_supported(const DmipMlp& net);
size_t surrogate_tc_workspace();
int launch_surrogate_tc(const DmipSurrogate* d, void* images, cudaStream_t s);
size_t metropolis_workspace(const DmipMetropolis* d);
int launch_metropolis(const DmipMetropolis* d, cudaStream_t s);
int launch_sample_t(const float* u, float* t, long long n, int debias, float beta_min, float beta_max, float t_epsilon,
                    float T, float eps_add, cudaStream_t s);
size_t sampler_tc_workspace();
void debug_set_timeline(unsigned long long* buf, int cap);
}  // namespace dmip
