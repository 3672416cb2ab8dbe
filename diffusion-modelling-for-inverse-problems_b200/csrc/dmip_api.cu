// dmip_api.cu — the extern "C" boundary of libdmip_sm100.so (declared in include/dmip.h).
// Validation mirrors the reference's own failure modes: shape asserts (nets.py:34, losses.py:79) and
// ValueError on bad option strings (losses.py:86,97; utils.py:31,46) become DMIP_EINVAL + a message.
#include "dmip_common.h"

namespace dmip {

static thread_local char g_err[512] = "";
static thread_local int g_launches = 0;

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches += n; }
void reset_launch_count() { g_launches = 0; }

int device_is_sm100() {
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return 0;
  return major == 10;
}

static int require_device() {
  if (!device_is_sm100()) {
    set_error("libdmip_sm100 needs an sm_100 (B200) device; there is no CPU or other-GPU fallback");
    return DMIP_EARCH;
  }
  return DMIP_OK;
}

static int check_sampler(const DmipSampler* d) {
  DMIP_REQUIRE(d != nullptr, "descriptor is NULL");
  DMIP_REQUIRE(d->variant == DMIP_CDE || d->variant == DMIP_CDIFFE || d->variant == DMIP_DPS,
               "No valid value for variant passed. Has to be one of DMIP_CDE, DMIP_CDIFFE or DMIP_DPS.");
  DMIP_REQUIRE(d->precision == DMIP_PREC_F32 || d->precision == DMIP_PREC_BF16, "unknown precision %d", d->precision);
  DMIP_REQUIRE(d->xdim >= 1 && d->ydim >= 1, "xdim/ydim must be positive");
  DMIP_REQUIRE(d->n_obs >= 0 && d->n_per_obs >= 0, "negative particle count");
  DMIP_REQUIRE(d->num_steps >= 1, "num_steps must be >= 1");
  DMIP_REQUIRE(d->sde_kind == DMIP_SDE_VP || d->sde_kind == DMIP_SDE_VE, "unknown sde_kind %d", d->sde_kind);
  DMIP_REQUIRE(d->sde_kind != DMIP_SDE_VE || (d->sigma_min > 0.f && d->sigma_max > d->sigma_min),
               "VE-SDE needs 0 < sigma_min < sigma_max");
  DMIP_REQUIRE(d->n_corrector >= 0 && d->n_corrector <= 8, "n_corrector must be in 0..8 (got %d)", d->n_corrector);
  DMIP_REQUIRE(d->n_corrector == 0 || d->snr > 0.f, "the corrector needs snr > 0");
  DMIP_REQUIRE(static_cast<long long>(d->num_steps) * (1 + d->n_corrector) < (1LL << 31), "too many sub-steps");
  DMIP_REQUIRE(d->rng_mode == DMIP_RNG_PHILOX || d->rng_mode == DMIP_RNG_INJECTED, "unknown rng_mode %d", d->rng_mode);
  if (d->n_obs > 0 && d->n_per_obs > 0) {
    DMIP_REQUIRE(d->y && d->out, "y / out is NULL");
    if (d->rng_mode == DMIP_RNG_INJECTED) {
      DMIP_REQUIRE(d->x0 && d->noise, "injected RNG mode needs x0 and noise");
      DMIP_REQUIRE(d->variant != DMIP_CDIFFE || d->ynoise, "injected RNG mode for CDiffE needs ynoise");
    }
  }
  const int want_in = d->xdim + d->ydim + 1;
  DMIP_REQUIRE(d->net.in_dim == want_in, "Input Tensor is expected to have xdim+ydim+1 = %d columns (net.in_dim = %d)",
               want_in, d->net.in_dim);
  if (d->variant == DMIP_CDIFFE)
    DMIP_REQUIRE(d->net.out_dim == d->xdim + d->ydim, "CDiffE net must output xdim+ydim columns");
  else
    DMIP_REQUIRE(d->net.out_dim == d->xdim, "net must output xdim columns");
  if (d->variant == DMIP_DPS)
    DMIP_REQUIRE(d->net2.in_dim == d->xdim + 1 && d->net2.out_dim == d->xdim, "prior_net must map [x,t] -> x");
  return DMIP_OK;
}

}  // namespace dmip

using namespace dmip;

extern "C" {

int dmip_version(void) { return DMIP_VERSION; }
const char* dmip_last_error(void) { return g_err; }
int dmip_device_ok(void) { return device_is_sm100(); }
int dmip_last_launch_count(void) { return g_launches; }

size_t dmip_pack_bytes(const DmipMlp* net, int32_t n_varying, int32_t out_rows, int32_t l0_split) {
  TcNetGeom g;
  if (tc_net_geom(net, n_varying, out_rows, l0_split, &g)) return 0;
  return g.bytes();
}

int dmip_pack_mlp(const DmipMlp* net, int32_t n_varying, int32_t out_rows, int32_t l0_split, void* packed,
                  size_t packed_bytes, void* stream) {
  reset_launch_count();
  int rc = require_device();
  if (rc) return rc;
  TcNetGeom g;
  if ((rc = tc_net_geom(net, n_varying, out_rows, l0_split, &g))) return rc;
  if (!packed || packed_bytes < g.bytes()) {
    set_error("packed buffer too small: need %zu bytes", g.bytes());
    return DMIP_EWORKSPACE;
  }
  DMIP_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 15) == 0, "packed buffer must be 16-byte aligned");
  return launch_pack(net, g, packed, static_cast<cudaStream_t>(stream));
}

size_t dmip_sampler_workspace_bytes(const DmipSampler* d) {
  if (!d) return 0;
  if (d->precision == DMIP_PREC_BF16) return sampler_tc_workspace();
  return sampler_f32_workspace(d);
}

int dmip_sampler_em_vp(const DmipSampler* d, void* stream) {
  reset_launch_count();
  int rc = require_device();
  if (rc) return rc;
  if ((rc = check_sampler(d))) return rc;
  if (d->n_obs == 0 || d->n_per_obs == 0) return DMIP_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (d->precision == DMIP_PREC_BF16) {
    DMIP_REQUIRE(d->packed != nullptr, "DMIP_PREC_BF16 needs a dmip_pack_mlp image in `packed`");
    return launch_sampler_tc(d, s);
  }
  if (d->workspace_bytes < sampler_f32_workspace(d) || !d->workspace) {
    set_error("workspace too small: need %zu bytes", sampler_f32_workspace(d));
    return DMIP_EWORKSPACE;
  }
  return launch_sampler_f32(d, s);
}

size_t dmip_forward_workspace_bytes(const DmipForward* d) {
  if (!d || d->precision != DMIP_PREC_F32) return 0;
  return forward_f32_workspace(d);
}

int dmip_mlp_forward(const DmipForward* d, void* stream) {
  reset_launch_count();
  int rc = require_device();
  if (rc) return rc;
  DMIP_REQUIRE(d != nullptr, "descriptor is NULL");
  DMIP_REQUIRE(d->n >= 0, "negative row count");
  DMIP_REQUIRE(d->x_dim + d->cond_dim + 1 == d->net.in_dim,
               "Input Tensor is expected to be 2D with x_dim+cond_dim+1 = %d columns (net.in_dim = %d)",
               d->x_dim + d->cond_dim + 1, d->net.in_dim);
  if (d->n == 0) return DMIP_OK;
  DMIP_REQUIRE(d->x && d->t && d->out && (d->cond || d->cond_dim == 0), "x / cond / t / out is NULL");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (d->precision == DMIP_PREC_BF16) {
    DMIP_REQUIRE(d->packed != nullptr, "DMIP_PREC_BF16 needs a dmip_pack_mlp image in `packed`");
    return launch_forward_tc(d, s);
  }
  DMIP_REQUIRE(d->precision == DMIP_PREC_F32, "unknown precision %d", d->precision);
  if (d->workspace_bytes < forward_f32_workspace(d) || !d->workspace) {
    set_error("workspace too small: need %zu bytes", forward_f32_workspace(d));
    return DMIP_EWORKSPACE;
  }
  return launch_forward_f32(d, s);
}

size_t dmip_loss_workspace_bytes(const DmipLoss* d) { return d ? loss_workspace(d) : 0; }
size_t dmip_loss_grad_floats(const DmipMlp* net) { return net ? loss_grad_floats(net) : 0; }

int dmip_loss_fwd_bwd(const DmipLoss* d, void* stream) {
  reset_launch_count();
  int rc = require_device();
  if (rc) return rc;
  DMIP_REQUIRE(d != nullptr, "descriptor is NULL");
  DMIP_REQUIRE(d->batch >= 0, "negative batch");
  return launch_loss(d, static_cast<cudaStream_t>(stream));
}

size_t dmip_mlp_grad_workspace_bytes(const DmipMlpGrad* d) { return d ? mlp_grad_workspace(d) : 0; }

int dmip_mlp_forward_stash(const DmipMlpGrad* d, void* stream) {
  reset_launch_count();
  int rc = require_device();
  if (rc) return rc;
  DMIP_REQUIRE(d != nullptr, "descriptor is NULL");
  return launch_mlp_forward_stash(d, static_cast<cudaStream_t>(stream));
}

int dmip_mlp_backward(const DmipMlpGrad* d, void* stream) {
  reset_launch_count();
  int rc = require_device();
  if (rc) return rc;
  DMIP_REQUIRE(d != nullptr, "descriptor is NULL");
  return launch_mlp_backward(d, static_cast<cudaStream_t>(stream));
}

size_t dmip_mlp_double_backward_workspace_bytes(const DmipMlpGradGrad* d) { return d ? mlp_double_backward_workspace(d) : 0; }

int dmip_mlp_double_backward(const DmipMlpGradGrad* d, void* stream) {
  reset_launch_count();
  int rc = require_device();
  if (rc) return rc;
  DMIP_REQUIRE(d != nullptr, "descriptor is NULL");
  return launch_mlp_double_backward(d, static_cast<cudaStream_t>(stream));
}

size_t dmip_surrogate_workspace_bytes(const DmipSurrogate* d) { return d ? surrogate_workspace(d) : 0; }

int dmip_surrogate_score(const DmipSurrogate* d, void* stream) {
  reset_launch_count();
  int rc = require_device();
  if (rc) return rc;
  DMIP_REQUIRE(d != nullptr, "descriptor is NULL");
  return launch_surrogate(d, static_cast<cudaStream_t>(stream));
}

size_t dmip_metropolis_workspace_bytes(const DmipMetropolis* d) { return d ? metropolis_workspace(d) : 0; }

int dmip_metropolis(const DmipMetropolis* d, void* stream) {
  reset_launch_count();
  int rc = require_device();
  if (rc) return rc;
  DMIP_REQUIRE(d != nullptr, "descriptor is NULL");
  return launch_metropolis(d, static_cast<cudaStream_t>(stream));
}

size_t dmip_posterior_loss_workspace_bytes(const DmipPosteriorLoss* d) { return d ? posterior_loss_workspace(d) : 0; }

int dmip_posterior_loss_fwd_bwd(const DmipPosteriorLoss* d, void* stream) {
  reset_launch_count();
  int rc = require_device();
  if (rc) return rc;
  DMIP_REQUIRE(d != nullptr, "descriptor is NULL");
  return launch_posterior_loss(d, static_cast<cudaStream_t>(stream));
}

int dmip_histogramdd(const DmipHistogram* d, void* stream) {
  reset_launch_count();
  int rc = require_device();
  if (rc) return rc;
  DMIP_REQUIRE(d != nullptr, "descriptor is NULL");
  return launch_histogramdd(d, static_cast<cudaStream_t>(stream));
}

int dmip_hist_kl(const void* hist_p, const void* hist_q, int64_t n_bins_total, double epsilon, double* out, void* stream) {
  reset_launch_count();
  int rc = require_device();
  if (rc) return rc;
  return launch_hist_kl(hist_p, hist_q, n_bins_total, epsilon, out, static_cast<cudaStream_t>(stream));
}

size_t dmip_mmd_workspace_bytes(const DmipMmd* d) { return mmd_workspace(d); }

int dmip_mmd(const DmipMmd* d, void* stream) {
  reset_launch_count();
  int rc = require_device();
  if (rc) return rc;
  DMIP_REQUIRE(d != nullptr, "descriptor is NULL");
  return launch_mmd(d, static_cast<cudaStream_t>(stream));
}

int dmip_sample_t(const float* u, float* t, int64_t n, int32_t debias, float beta_min, float beta_max, float t_epsilon,
                  float T, float eps_add, void* stream) {
  reset_launch_count();
  int rc = require_device();
  if (rc) return rc;
  return launch_sample_t(u, t, n, debias, beta_min, beta_max, t_epsilon, T, eps_add, static_cast<cudaStream_t>(stream));
}

#if defined(DMIP_DEBUG) || defined(DMIP_JOBMARKS)
void dmip_debug_set_timeline(void* device_buf, int32_t capacity) {
  debug_set_timeline(static_cast<unsigned long long*>(device_buf), capacity);
}
#endif

}  // extern "C"
