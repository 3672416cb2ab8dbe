/*
 * dmip.h — C ABI of libdmip_sm100.so, the B200 (sm_100a) hot path of
 * maffos/Diffusion-Modelling-for-inverse-problems.
 *
 * The reference is pure Python/PyTorch and has NO plugin / FFI boundary
 * (SURVEY.md §8b): its "API that stays as it is" is the Python class surface of
 * models/diffusion.py, sdes.py, losses.py and nets.py.  This header is the new
 * boundary a maintainer binds underneath those classes (ctypes stub in
 * INTEGRATION.md).  Each entry point names the reference code it replaces.
 *
 * Conventions
 *   - plain C types only; every pointer marked "device" is a CUDA device pointer
 *     owned by the caller (e.g. a torch tensor's data_ptr()); the library never
 *     allocates or frees device memory and keeps no pointer after returning;
 *   - all work is enqueued on the cudaStream_t passed as `stream` (as void*),
 *     asynchronously, without internal synchronisation;
 *   - return value 0 = ok, negative = DMIP_E*; dmip_last_error() gives the
 *     message for the calling thread; no C++ exception crosses the boundary;
 *   - fp32 row-major contiguous tensors unless a leading dimension is given;
 *   - weights are nn.Linear layout: W (out_features, in_features), b (out_features).
 */
#ifndef DMIP_H_
#define DMIP_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DMIP_VERSION 100

#define DMIP_OK 0
#define DMIP_EINVAL (-1)     /* bad argument (reference: ValueError / assert, losses.py:79,86,97; nets.py:34) */
#define DMIP_EARCH (-2)      /* device is not sm_100 */
#define DMIP_EWORKSPACE (-3) /* workspace too small; see dmip_*_workspace_bytes */
#define DMIP_ECUDA (-4)      /* CUDA runtime error; message carries cudaGetErrorString */

#define DMIP_MAX_LAYERS 8

/* precision of the score-net evaluation */
#define DMIP_PREC_F32 0  /* fp32 FFMA kernels: any layer widths; matches the reference to fp32 round-off  */
#define DMIP_PREC_BF16 1 /* tcgen05 kernels: bf16 operands / fp32 accumulate; hidden_layers == [512,512,512] */

/* sampler variants: models/diffusion.py classes */
#define DMIP_CDE 0    /* CDE  — BaseClassDiffusionModel.forward, models/diffusion.py:27-46                  */
#define DMIP_CDIFFE 1 /* CDiffE.forward, models/diffusion.py:158-180 (with the `cond` fix, SURVEY.md Q7)    */
#define DMIP_DPS 2    /* PosteriorDiffusionEstimator: base forward with nets.py:155-157 PosteriorScore as a */

#define DMIP_SDE_VP 0 /* VariancePreservingSDE, sdes.py:9-57                                                       */
#define DMIP_SDE_VE 1 /* variance-exploding SDE (no upstream counterpart)                                         */

#define DMIP_RNG_PHILOX 0   /* counter-based Philox4x32-10 keyed by global particle index                  */
#define DMIP_RNG_INJECTED 1 /* caller supplies x0 / per-step noise (parity tests, SURVEY.md Q6)            */

/* A tanh MLP as built by nets.py:17-30 (MLP / MLP2): n_layers Linear layers, tanh after every layer but the
 * last, and tanh applied TWICE after layer 0 (the Sequential 'act' quirk, SURVEY.md Q1). */
typedef struct DmipMlp {
  int32_t n_layers; /* number of nn.Linear layers (= len(hidden_layers)+1), 2..DMIP_MAX_LAYERS   */
  int32_t in_dim;   /* columns of cat[x, cond, t]                                                 */
  int32_t out_dim;
  int32_t width[DMIP_MAX_LAYERS]; /* out_features of layer l (width[n_layers-1] == out_dim)       */
  const float* W[DMIP_MAX_LAYERS]; /* device, (width[l], width[l-1] or in_dim)                     */
  const float* b[DMIP_MAX_LAYERS]; /* device, (width[l],)                                          */
} DmipMlp;

int dmip_version(void);
const char* dmip_last_error(void);
/* 1 if the current device can run the library (compute capability 10.x), else 0 */
int dmip_device_ok(void);

/* ---- weight packing for the tcgen05 path -------------------------------------------------------------
 * Re-tiles one net into the bf16, 128B-swizzled, K-major stage images the sampler streams with bulk-TMA.
 * `n_varying` = leading input columns that vary per row and therefore enter the layer-0 GEMM (the rest —
 * y and/or t — are folded into an fp32 per-step bias by the kernel); `out_rows` = leading output rows kept
 * (CDiffE needs only the first xdim outputs, models/diffusion.py:177); `l0_split` in {1,2,3,4}: layer-0
 * operand splitting (1: bf16 x; 2: x = hi+lo, both bf16; 3: also W0 = hi+lo; 4: ONE f16 part — layer 0 is an f16 x f16
 * product, 11 mantissa bits of the state at the MMA count of mode 1: as accurate as mode 2 in every sampler test
 * because the bf16 hidden layers dominate the error, and 6 % faster; the Python classes default to it).  Call again after every
 * optimizer.step().  Replaces nothing in the reference (its weights are read in place by addmm). */
size_t dmip_pack_bytes(const DmipMlp* net, int32_t n_varying, int32_t out_rows, int32_t l0_split);
int dmip_pack_mlp(const DmipMlp* net, int32_t n_varying, int32_t out_rows, int32_t l0_split, void* packed,
                  size_t packed_bytes, void* stream);

/* ---- reverse-SDE Euler–Maruyama posterior sampler -----------------------------------------------------
 * Replaces the S-step loop of models/diffusion.py:38-42 / :171-177 together with sdes.py:77-87 (mu, sigma),
 * sdes.py:21-35 (beta, f, g), sdes.py:37-49 (CDiffE re-diffusion of y) and nets.py:32-35/52-57/155-157.
 * One call integrates n_obs * n_per_obs particles for num_steps steps; particles of observation o occupy
 * rows [o*n_per_obs, (o+1)*n_per_obs) of every per-particle tensor.
 *
 * Shapes each kernel family serves (outside them dmip_sampler_em_vp returns DMIP_EINVAL and names the limit):
 *   DMIP_PREC_BF16 (tcgen05, the state lives in registers as 8-column pieces): hidden layers [512,512,512] and
 *     CDE xdim <= 104; CDiffE xdim <= 32 and ydim <= 24; DPS xdim <= 8 (both nets);
 *     the layer-0 GEMM depth of dmip_pack_bytes (the varying columns, split l0_split ways) at most 512.
 *   DMIP_PREC_F32 (FFMA): 2..DMIP_MAX_LAYERS Linear layers of widths 1..512 (in_dim too), and DPS xdim <= 128.
 * The Python classes (models/diffusion.py) run precision='bf16' on the FFMA kernels where the tcgen05 limits are not
 * met and record the path that ran in `last_precision`. */
typedef struct DmipSampler {
  int32_t variant;   /* DMIP_CDE / DMIP_CDIFFE / DMIP_DPS                                          */
  int32_t precision; /* DMIP_PREC_*                                                                 */
  int32_t xdim, ydim;
  int32_t n_obs;
  int64_t n_per_obs;
  int32_t num_steps;               /* S; reference default 200 (models/diffusion.py:27)            */
  float T, beta_min, beta_max;     /* sdes.py:14-19 defaults 1, 0.1, 20                             */
  float mean, std;                 /* x0 = randn*std + mean (models/diffusion.py:32-33)             */
  DmipMlp net;                     /* CDE/CDiffE: sde.a ; DPS: likelihood_net (MLP on [x,y,t])      */
  DmipMlp net2;                    /* DPS only: prior_net (MLP2 on [x,t])                           */
  const void* packed;              /* DMIP_PREC_BF16: dmip_pack_mlp image of `net`                   */
  const void* packed2;             /* DMIP_PREC_BF16 + DPS: image of `net2`                          */
  int32_t l0_split;                /* must equal the value given to dmip_pack_mlp                    */
  const float* y;                  /* device (n_obs, ydim)                                           */
  float* out;                      /* device (n_obs*n_per_obs, xdim): final x_t (also the fp32 state)*/
  int32_t rng_mode;                /* DMIP_RNG_*                                                     */
  uint64_t seed;                   /* Philox key                                                     */
  uint64_t gidx_base;              /* global index of this call's particle 0 (multi-GPU sharding)    */
  const float* x0;                 /* injected: (n_obs*n_per_obs, xdim) standard normals             */
  const float* noise;              /* injected: (S, n_obs*n_per_obs, xdim)                           */
  const float* ynoise;             /* injected, CDiffE: (S, n_obs*n_per_obs, ydim)                   */
  void* workspace;                 /* device scratch, dmip_sampler_workspace_bytes(), 16-byte aligned */
  size_t workspace_bytes;
  /* ---- beyond the reference (all zero = the reference's sampler: VP-SDE, Euler–Maruyama predictor only).
   * BASELINE.json names "VP/VE SDE" and a "predictor sampler"; upstream has only VP (sdes.py:9-57) and no corrector, so
   * these have no reference counterpart (parity unpinned; oracle restatement: oracle/sampler.py pc_sampler).
   * VE: sigma(t) = sigma_min (sigma_max / sigma_min)^t, f = 0, g = sigma sqrt(2 ln(sigma_max / sigma_min)) (Song et al.
   * 2021); CDiffE re-diffuses y with x_t | x_0 ~ N(x_0, sigma(t)^2).  n_corrector Langevin sub-steps follow every
   * predictor step at its new time level: x += e s + sqrt(2 e) z, e = 2 snr^2 std(t)^2 (closed form of Song's norm rule).
   * With correctors the sub-step index u = step * (1 + n_corrector) + c is the Philox step key and the first index of
   * the injected noise / ynoise tensors, which then hold num_steps * (1 + n_corrector) slices. */
  int32_t sde_kind;                /* DMIP_SDE_VP (0) / DMIP_SDE_VE (1)                               */
  float sigma_min, sigma_max;      /* VE only                                                         */
  int32_t n_corrector;             /* Langevin corrector sub-steps per step, 0..8                     */
  float snr;                       /* corrector signal-to-noise ratio (Song et al.: 0.16)             */
} DmipSampler;

size_t dmip_sampler_workspace_bytes(const DmipSampler* d);
int dmip_sampler_em_vp(const DmipSampler* d, void* stream);
/* number of kernel launches the last dmip_* call on this thread enqueued (bench.py's gpu_launches) */
int dmip_last_launch_count(void);

/* ---- score-net forward  a(x, cond, t) ------------------------------------------------------------------
 * Replaces MLP.forward / MLP2.forward (nets.py:32-35, :52-57): cat[x, cond, t] -> net.  `cond` may be NULL
 * with cond_dim 0 (MLP2, or the empty tensor of losses.py:149).  out: (n, net.out_dim). */
typedef struct DmipForward {
  int32_t precision;
  DmipMlp net;
  const void* packed; /* DMIP_PREC_BF16: image packed with n_varying = in_dim, out_rows = out_dim */
  int32_t l0_split;
  int64_t n;
  int32_t x_dim, cond_dim;
  const float* x;    /* device (n, x_dim)    */
  const float* cond; /* device (n, cond_dim) */
  const float* t;    /* device (n,)          */
  float* out;        /* device (n, out_dim)  */
  void* workspace;
  size_t workspace_bytes;
} DmipForward;

size_t dmip_forward_workspace_bytes(const DmipForward* d);
int dmip_mlp_forward(const DmipForward* d, void* stream);

/* ---- score-net forward WITH a backward: autograd support for user-written losses --------------------------------
 * dmip_mlp_forward_stash evaluates a(x, cond, t) like dmip_mlp_forward and keeps, in the caller's workspace, what the
 * backward needs; dmip_mlp_backward turns a gradient w.r.t. the outputs into the flat parameter gradient
 * [W_0, b_0, W_1, b_1, ...] and (optionally) the gradient w.r.t. the concatenated inputs cat[x, cond, t] — what
 * `out.backward()` does through nets.py:32-35 / :52-57 upstream.  tcgen05 kernels, bf16x3 split products (fp32-level
 * accuracy); nets [in <= 64] -> 512 -> 512 -> 512 -> [out <= 64] only (dmip_mlp_grad_workspace_bytes returns 0 otherwise and
 * the Python layer falls back to the plain torch module chain with a warning).  The same descriptor (same workspace,
 * untouched in between) must be passed to both calls; first-order derivatives only. */
typedef struct DmipMlpGrad {
  DmipMlp net;
  int64_t n;
  int32_t x_dim, cond_dim;
  const float* x;          /* device (n, x_dim)                       */
  const float* cond;       /* device (n, cond_dim) or NULL            */
  const float* t;          /* device (n,)                             */
  float* out;              /* forward:  device (n, out_dim)           */
  const float* grad_out;   /* backward: device (n, out_dim)           */
  float* grad_params;      /* backward: device float[dmip_loss_grad_floats(net)], overwritten */
  float* grad_in;          /* backward: device (n, in_dim) or NULL    */
  void* workspace;         /* device, dmip_mlp_grad_workspace_bytes(), 1024-byte aligned; lives from forward to backward */
  size_t workspace_bytes;
} DmipMlpGrad;

size_t dmip_mlp_grad_workspace_bytes(const DmipMlpGrad* d);
int dmip_mlp_forward_stash(const DmipMlpGrad* d, void* stream);
int dmip_mlp_backward(const DmipMlpGrad* d, void* stream);

/* ---- fused score-training losses: forward + backward in one call -------------------------------------------
 * Replaces, per batch, the body of CDE/CDiffE.train_epoch (models/diffusion.py:80-88, :129-139) up to and including
 * loss.backward(): VariancePreservingSDE.sample with the Gaussian draw `eps` supplied by the caller, the net
 * evaluations, DSMLoss (losses.py:49-52), ScoreFPELoss with exact divergence (losses.py:77-98),
 * ConditionalScoreFPELoss (losses.py:116-124), DSM_PDELoss (losses.py:143-164), PINNLoss (losses.py:214-242).
 * Outputs: out_losses[4] = {loss, mean DSM, mean initial-condition (x lam2), mean PDE (x lam)} — the reference's
 * return value and info dict — and d loss / d parameters in `grad`, flat fp32 [W_0, b_0, W_1, b_1, ...] (both are
 * overwritten).  Means divide by batch_global (>= batch; data-parallel ranks pass the global batch and all-reduce
 * `grad` and `out_losses` with SUM).  fp32 FFMA kernels, any layer widths <= 512. */
#define DMIP_LOSS_DSM 0     /* loss_fn.name == 'DSMLoss'                                   */
#define DMIP_LOSS_DSM_PDE 1 /* DSM_PDELoss                                                 */
#define DMIP_LOSS_PINN 2    /* PINNLoss                                                    */
#define DMIP_LOSS_PINN2 3   /* PINNLoss2 (losses.py:245-291): PINNLoss WITHOUT the DSM term in the objective — total =
                               lam2 ic + lam pde; out_losses[1] still reports the mean DSM loss (its 'DSM_eval' entry)  */
#define DMIP_PDE_FPE 0      /* pde_loss = 'FPE'  (exact divergence: d = xdim [+ydim for CDiffE] <= 31) */
#define DMIP_PDE_CFPE 1     /* pde_loss = 'cScoreFPE'                                      */
/* divergence_method of ScoreFPELoss.forward (losses.py:81-86).  EXACT: d <= 4 runs forward-only (d + d(d+1)/2 tangent
 * streams), larger d takes the adjoint route (d tangent streams forward, one reverse sweep for grad_x);
 * EXACT_ADJOINT forces the adjoint route (same values; test hook); HUTCHINSON: v.(J v) with the caller's probe. */
#define DMIP_DIV_EXACT 0
#define DMIP_DIV_HUTCHINSON 1
#define DMIP_DIV_EXACT_ADJOINT 2
#define DMIP_L1 1
#define DMIP_L2 2

typedef struct DmipLoss {
  int32_t kind;  /* DMIP_LOSS_*                      */
  int32_t model; /* DMIP_CDE or DMIP_CDIFFE          */
  int32_t xdim, ydim;
  int64_t batch;
  int64_t batch_global; /* 0 = batch */
  DmipMlp net;          /* sde.a */
  float beta_min, beta_max;
  float lam, lam2;
  int32_t pde_loss, pde_metric, ic_metric;
  int32_t divergence;     /* DMIP_DIV_*: ScoreFPELoss.forward's divergence_method (losses.py:77-86)                  */
  const float* x;         /* device (batch, xdim)                                           */
  const float* y;         /* device (batch, ydim)                                           */
  const float* t;         /* device (batch,)  from sample_t (models/diffusion.py:48-58)     */
  const float* eps;       /* device (batch, d) standard normals, d = xdim (CDE) | xdim+ydim */
  const float* ic_target; /* device (batch, xdim) = initial_condition(x, y); PINN only      */
  const float* hutch_v;   /* device (batch, d) probe of div_estimator (losses.py:28-40): +-1 (rademacher_like) or
                             Gaussian; DMIP_DIV_HUTCHINSON only                              */
  float* out_losses;      /* device float[4]                                                */
  float* grad;            /* device float[dmip_loss_grad_floats(net)]                       */
  void* workspace;        /* device, dmip_loss_workspace_bytes(), 16-byte aligned           */
  size_t workspace_bytes;
} DmipLoss;

size_t dmip_loss_workspace_bytes(const DmipLoss* d);
size_t dmip_loss_grad_floats(const DmipMlp* net);
int dmip_loss_fwd_bwd(const DmipLoss* d, void* stream);

/* ---- scatterometry surrogate: energy / posterior score / likelihood VJP (K4) ----------------------------------
 * The frozen forward model f: R^3 -> R^23 is the ReLU MLP of utils_scatterometry.py:9-16 (surrogate.pt; relu after
 * every layer but the last).  One call runs forward + reverse sweep through it for n rows.
 *   mode DMIP_SURR_ENERGY   energy[i] = get_log_posterior(x_i, f, a, b, y_i, lambd_bd)  (utils_scatterometry.py:30-38)
 *                           grad[i]   = d energy / d x_i = energy_grad (models/SNF.py:234-237);
 *                           score_posterior = -grad is the PINNLoss initial condition
 *                           (main_diffusion_scatterometry.py:142-145) and the drift of the Metropolis reference chain.
 *   mode DMIP_SURR_LIK_VJP  grad[i] = J_f(x_i)^T (-a^2 v1 + v2 + a^2 v3), the three surrogate VJPs of
 *                           PosteriorLoss.likelihood_target (losses.py:349-371) merged; `energy` unused.
 * fx (optional): f(x) (n, out_dim).  Any widths <= 512, 2..DMIP_MAX_LAYERS layers.
 * Nets of the reference's surrogate shape — [in <= 3] -> 256 -> 256 -> 256 -> [out <= 32] — run the tcgen05 kernel
 * (csrc/dmip_surrogate_tc.cu: bf16x3 split products, fp32 accumulate: f to ~5e-6 relative, energy and gradient within 2e-4;
 * the gradient of a row within rounding distance of a ReLU kink may take the other side's value), every other net the
 * fp32 FFMA kernel; DMIP_SURROGATE_PATH=ffma in the environment forces the FFMA kernel. */
#define DMIP_SURR_ENERGY 0
#define DMIP_SURR_LIK_VJP 1

typedef struct DmipSurrogate {
  int32_t mode;
  DmipMlp net;          /* the surrogate (ReLU MLP), in_dim = xdim, out_dim = ydim                    */
  float a, b, lambd_bd; /* noise model p = (a f)^2 + b^2 and boundary weight (utils_scatterometry.py:19-21) */
  int64_t n;
  const float* x;       /* device (n, in_dim)  */
  const float* y;       /* device (n, out_dim), or (ceil(n / rows_per_obs), out_dim) when rows_per_obs > 0 */
  float* energy;        /* device (n,) or NULL */
  float* grad;          /* device (n, in_dim)  */
  float* fx;            /* device (n, out_dim) or NULL */
  void* workspace;      /* device, dmip_surrogate_workspace_bytes() */
  size_t workspace_bytes;
  int64_t rows_per_obs; /* 0: y holds n rows, one per row of x.  > 0: row i belongs to observation i / rows_per_obs and y
                           holds ceil(n / rows_per_obs) rows — batches of n_obs x n_per_obs rows laid out as DmipSampler
                           lays out its particles; rows_per_obs = n is the reference's broadcast of ONE observation
                           over all samples (utils_scatterometry.py:30-38 with ys of shape (1, ydim)) */
} DmipSurrogate;

size_t dmip_surrogate_workspace_bytes(const DmipSurrogate* d);
int dmip_surrogate_score(const DmipSurrogate* d, void* stream);

/* ---- Metropolis ground-truth chains on the scatterometry posterior ---------------------------------------------
 * Replaces anneal_to_energy (models/SNF.py:250-275, langevin_prop=False) as generate_gt_samples calls it
 * (generate_scatterometry_ground_truth.py:26-29): `steps` random-walk Metropolis steps on E = get_log_posterior,
 * proposal x + noise_std * N(0, I), accept when u < exp(E(x) - E(x')).  n_obs * n_per_obs independent chains, chain i
 * targets observation y[i / n_per_obs]; x holds the start points on entry (upstream: U(-1,1)^3) and the final points on
 * return; de (optional) = E(final) - E(start), the second return value of anneal_to_energy.  One launch runs all steps.
 * rng_mode DMIP_RNG_PHILOX: in-kernel Philox keyed by (seed, gidx_base + chain, step); DMIP_RNG_INJECTED: the caller's
 * normals noise (steps, n, xdim) and uniforms unif (steps, n), in the order the reference draws them. */
typedef struct DmipMetropolis {
  DmipMlp net;             /* the surrogate (ReLU MLP), in_dim = xdim <= 8, out_dim = ydim */
  float a, b, lambd_bd;
  float noise_std;         /* NOISE_STD_MCMC */
  int32_t n_obs;
  int64_t n_per_obs;
  int32_t steps;           /* METR_STEPS */
  const float* y;          /* device (n_obs, ydim) */
  float* x;                /* device (n_obs * n_per_obs, xdim), in/out */
  float* de;               /* device (n_obs * n_per_obs,) or NULL */
  int32_t rng_mode;
  uint64_t seed, gidx_base;
  const float* noise;
  const float* unif;
  void* workspace;         /* device, dmip_metropolis_workspace_bytes() */
  size_t workspace_bytes;
} DmipMetropolis;

size_t dmip_metropolis_workspace_bytes(const DmipMetropolis* d);
int dmip_metropolis(const DmipMetropolis* d, void* stream);

/* ---- PosteriorLoss (DPS joint loss), forward + backward -------------------------------------------------------
 * Replaces PosteriorLoss.forward + likelihood_target (losses.py:349-386) and the loss.backward() of
 * PosteriorDiffusionEstimator.train_epoch (models/diffusion.py:204-229):
 *   prior_loss = DSM(prior_net(x_t,t), std, eps);  x0_hat = (x_t + std^2 s_prior)/alpha;
 *   target = (std^2 J_s^T + I) J_f(x0_hat)^T (-a^2 v1 + v2 + a^2 v3)   (constant in the backward pass: the reference
 *   calls autograd.grad without create_graph);  lik_loss = sum_j (alpha s_lik - target)^2;
 *   loss = mean(prior_loss + lam * lik_loss).
 * out_losses[4] = {loss, mean prior_loss, lam * mean lik_loss, 0}; grad_prior / grad_lik: flat fp32 gradients of the
 * two nets ([W_0,b_0,W_1,b_1,...]).  J_s comes from xdim forward-mode tangent streams through the prior net. */
typedef struct DmipPosteriorLoss {
  int32_t xdim, ydim;
  int64_t batch;
  int64_t batch_global;   /* 0 = batch */
  DmipMlp prior_net;      /* MLP2 on [x_t, t]      */
  DmipMlp lik_net;        /* MLP  on [x_t, y, t]   */
  DmipMlp surrogate;      /* forward model f       */
  float beta_min, beta_max;
  float a, b, lam;
  const float* x;         /* device (batch, xdim)  */
  const float* y;         /* device (batch, ydim)  */
  const float* t;         /* device (batch,)       */
  const float* eps;       /* device (batch, xdim)  */
  float* out_losses;      /* device float[4]       */
  float* grad_prior;      /* device float[dmip_loss_grad_floats(prior_net)] */
  float* grad_lik;        /* device float[dmip_loss_grad_floats(lik_net)]   */
  void* workspace;
  size_t workspace_bytes;
} DmipPosteriorLoss;

size_t dmip_posterior_loss_workspace_bytes(const DmipPosteriorLoss* d);
int dmip_posterior_loss_fwd_bwd(const DmipPosteriorLoss* d, void* stream);

/* ---- evaluation metrics next to the sampler (SURVEY.md §8f N2) ------------------------------------------------------
 * dmip_histogramdd: np.histogramdd(x, bins, range) of main_diffusion_linear.py:85-88 /
 * main_diffusion_scatterometry.py:72-75, bit-exact (per dimension searchsorted(edges, x, 'right') - 1, last edge
 * inclusive, out-of-range samples dropped); `counts` (uint64, prod(bins), C order) is ACCUMULATED into, which is the
 * reference's `hist_sum += hist` over repeats.  edges[d]: device double[bins[d] + 1] (np.linspace(lo, hi, bins + 1)).
 * dmip_hist_kl: sum(rel_entr(p, q)) with the reference's normalisation (h / sum, + epsilon, / sum;
 * main_diffusion_linear.py:108-116): out = device double[3] {KL, sum(hp), sum(hq)}. */
typedef struct DmipHistogram {
  int32_t dim;               /* 1..4                         */
  int32_t bins[4];
  const double* edges[4];    /* device                       */
  int64_t n;
  const float* x;            /* device (n, dim)              */
  void* counts;              /* device uint64[prod(bins)]    */
} DmipHistogram;

int dmip_histogramdd(const DmipHistogram* d, void* stream);
int dmip_hist_kl(const void* hist_p, const void* hist_q, int64_t n_bins_total, double epsilon, double* out, void* stream);

/* ---- unbiased Gaussian-kernel MMD^2 between posterior sample sets ---------------------------------------------------
 * No reference counterpart (the reference reports only the histogram KL above).  The estimator is MMD^2_u of
 * Gretton et al. 2012 (JMLR 13, eq. 3): per observation o and bandwidth b, with k(a, c) = exp(-|a - c|^2 / (2 sigma_b^2)),
 *   Kxx = mean_{i != j} k(x_i, x_j),  Kyy = mean_{i != j} k(y_i, y_j),  Kxy = mean_{i, j} k(x_i, y_j),
 *   MMD^2_u = Kxx + Kyy - 2 Kxy;
 * out[o][b] = {MMD^2_u, Kxx, Kyy, Kxy} (float64).  Distances and kernel values are fp32 (ex2.approx), every sum that
 * leaves a thread is fp64.  Two launches per call; results are bit-identical from run to run on one device.  The
 * workspace size depends on n_obs and n_bw only (< 100 KB + 24 B per observation and bandwidth). */
#define DMIP_MMD_MAX_DIM 16
#define DMIP_MMD_MAX_BW 8
typedef struct DmipMmd {
  int32_t dim;                  /* 1..DMIP_MMD_MAX_DIM                                          */
  int32_t n_obs;                /* >= 1                                                          */
  int64_t n, m;                 /* samples per observation in x / y, each >= 2                   */
  int32_t n_bw;                 /* 1..DMIP_MMD_MAX_BW                                            */
  float sigma[DMIP_MMD_MAX_BW]; /* k(a,b) = exp(-|a-b|^2 / (2 sigma^2)), sigma > 0 and finite    */
  const float* x;               /* device (n_obs, n, dim)                                        */
  const float* y;               /* device (n_obs, m, dim)                                        */
  double* out;                  /* device (n_obs, n_bw, 4): {MMD^2_u, Kxx, Kyy, Kxy}             */
  void* workspace;              /* device, dmip_mmd_workspace_bytes(), 8-byte aligned            */
  size_t workspace_bytes;
} DmipMmd;

size_t dmip_mmd_workspace_bytes(const DmipMmd* d);
int dmip_mmd(const DmipMmd* d, void* stream);

/* ---- training-time draw of t on the device ---------------------------------------------------------------------------
 * BaseClassDiffusionModel.sample_t (models/diffusion.py:48-58): t[i] from the uniform u[i] (both device float[n]).
 * debias != 0: the inverse CDF of VariancePreservingSDE.sample_debiasing_t (sdes.py:51-57; q(t) ~ beta(t)/var(t),
 * constant below t_epsilon), then + eps_add, minus eps_add again where the sum exceeds T; debias == 0: eps_add + u T,
 * clamped to T - eps_add.  The reference draws on the CPU and copies t over every batch. */
int dmip_sample_t(const float* u, float* t, int64_t n, int32_t debias, float beta_min, float beta_max, float t_epsilon,
                  float T, float eps_add, void* stream);

/* ---- debug hook (exists only in -DDMIP_DEBUG / -DDMIP_JOBMARKS builds of the library; the tcgen05 building-block
 * self-tests and micro-benchmarks live in tools/probe/, outside the product) ------------------------------------------
 * Timeline: when set, CTA 0 of the tcgen05 sampler records (clock64 << 16 | event code) entries into
 * device_buf[1..capacity) and the entry count into device_buf[0] (uint64).  Pass NULL to switch off. */
#if defined(DMIP_DEBUG) || defined(DMIP_JOBMARKS)
void dmip_debug_set_timeline(void* device_buf, int32_t capacity);
#endif

#ifdef __cplusplus
}
#endif
#endif /* DMIP_H_ */
