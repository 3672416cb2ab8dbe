"""Drop-in for the reference's `sdes.py` (VariancePreservingSDE :9-57, PluginReverseSDE :60-87).

Same class names, constructor arguments, attributes and method signatures.  The closed forms below are only the
*interface* (callers such as losses and evaluation scripts use them on small tensors); inside the sampler and the
fused losses the same formulas are evaluated in-kernel (csrc/dmip_tc.cu, csrc/dmip_f32.cu).  The reference's dead
methods `dsm` / `elbo_random_t_slice` (wrong arity, SURVEY.md App. C) are not carried over.
"""
import math

import torch


def vp_truncated_inverse_cdf(u, beta_min, beta_max, t_epsilon, T):
    """Inverse CDF of q(t) ∝ beta(t)/var(t), constant below t_epsilon — the distribution behind the reference's
    `sample_vp_truncated_q` (sdes.py:57; the implementation lives in the un-vendored sdeflow-light, so this is
    restated from its published form, SURVEY.md App. A.2)."""
    db = beta_max - beta_min

    def big_b(t):
        return 0.5 * t * t * db + t * beta_min

    def antider(t):
        b = big_b(t)
        return math.log(1.0 - math.exp(-b)) + b

    r_eps = (beta_min + db * t_epsilon) / (1.0 - math.exp(-big_b(t_epsilon)))
    a_eps = antider(t_epsilon)
    Z = r_eps * t_epsilon + antider(float(T)) - a_eps
    lin = Z / r_eps * u
    nl = (-beta_min + torch.sqrt(beta_min ** 2 + 2.0 * db * torch.log1p(torch.exp(Z * u + a_eps - r_eps * t_epsilon)))) / db
    return torch.where(u <= t_epsilon * r_eps / Z, lin, nl)


class VariancePreservingSDE(torch.nn.Module):
    """VP-SDE of Song et al. 2021: dy = -beta(t)/2 y dt + sqrt(beta(t)) dW."""

    def __init__(self, beta_min=0.1, beta_max=20.0, T=1.0, t_epsilon=0.001):
        super().__init__()
        self.beta_min = beta_min
        self.beta_max = beta_max
        self.T = T
        self.t_epsilon = t_epsilon

    def beta(self, t):
        return self.beta_min + (self.beta_max - self.beta_min) * t

    def _int_beta(self, t):
        return 0.5 * t ** 2 * (self.beta_max - self.beta_min) + t * self.beta_min

    def mean_weight(self, t):
        return torch.exp(-0.5 * self._int_beta(t))

    def var(self, t):
        return 1. - torch.exp(-self._int_beta(t))

    def f(self, t, y):
        return -0.5 * self.beta(t) * y

    def g(self, t, y):
        return torch.ones_like(y) * self.beta(t) ** 0.5

    def sample(self, t, y0, return_noise=False):
        """y_t | y_0; with return_noise also (epsilon, std, g) as the losses need them."""
        std = self.var(t) ** 0.5
        epsilon = torch.randn_like(y0)
        yt = epsilon * std + self.mean_weight(t) * y0
        if not return_noise:
            return yt
        return yt, epsilon, std, self.g(t, yt)

    def sample_debiasing_t(self, shape):
        """t ~ q(t) ∝ g²/std² truncated at t_epsilon (importance sampling that removes the DSM weight)."""
        u = torch.rand(*shape)
        return vp_truncated_inverse_cdf(u.view(-1), self.beta_min, self.beta_max, self.t_epsilon, self.T).view(*shape)

    def sample_t_device(self, shape, device, debias=True, eps=1e-4):
        """`sample_t` of the models (models/diffusion.py:48-58: the draw above + eps, folded back where it exceeds T; or
        eps + u T without debiasing) entirely on `device`: one torch.rand and one kernel (`dmip_sample_t`) instead of ten
        CPU ops and a host-to-device copy per batch.  Same distribution, the CUDA generator's stream."""
        import ctypes as C
        from . import _lib
        L = _lib.require_gpu()
        if not getattr(L, '_sample_t_bound', False):
            L.dmip_sample_t.restype = C.c_int
            L.dmip_sample_t.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_float, C.c_float,
                                        C.c_float, C.c_float, C.c_void_p]
            L._sample_t_bound = True
        u = torch.rand(*shape, device=device, dtype=torch.float32)
        t = torch.empty_like(u)
        with torch.cuda.device(device):
            _lib.check(L.dmip_sample_t(u.data_ptr(), t.data_ptr(), u.numel(), 1 if debias else 0, float(self.beta_min),
                                       float(self.beta_max), float(self.t_epsilon), float(self.T), float(eps),
                                       _lib.stream_ptr()))
        return t


class VarianceExplodingSDE(torch.nn.Module):
    """VE-SDE of Song et al. 2021 (eq. 30-31): dy = sqrt(d[sigma^2(t)]/dt) dW, sigma(t) = sigma_min (sigma_max/sigma_min)^t.

    NOT part of the reference (upstream ships only the VP-SDE, sdes.py:9-57); BASELINE.json names "VP/VE SDE", so this
    class carries the interface of `VariancePreservingSDE` (f, g, mean_weight, var, sample, sample_debiasing_t,
    sample_t_device) and the models accept it as `base_sde` (SURVEY.md §8f N4, parity unpinned; oracle restatements:
    oracle/ve.py, oracle/ve_losses.py).  Sampling, incl. the Langevin corrector, and the fused training losses (DSM,
    DSM_PDE, PINN, PINN2, PosteriorLoss) run in the same kernels as for the VP-SDE."""

    def __init__(self, sigma_min=0.01, sigma_max=50.0, T=1.0, t_epsilon=1e-5):
        super().__init__()
        self.sigma_min = sigma_min
        self.sigma_max = sigma_max
        self.T = T
        self.t_epsilon = t_epsilon
        # attribute names the samplers read from any base SDE
        self.beta_min = 0.0
        self.beta_max = 0.0

    def sigma(self, t):
        return self.sigma_min * (self.sigma_max / self.sigma_min) ** t

    def mean_weight(self, t):
        return torch.ones_like(t) if torch.is_tensor(t) else 1.0

    def var(self, t):
        return self.sigma(t) ** 2

    def f(self, t, y):
        return torch.zeros_like(y)

    def g(self, t, y):
        return torch.ones_like(y) * self.sigma(t) * math.sqrt(2.0 * math.log(self.sigma_max / self.sigma_min))

    def sample(self, t, y0, return_noise=False):
        std = self.var(t) ** 0.5
        epsilon = torch.randn_like(y0)
        yt = epsilon * std + y0
        if not return_noise:
            return yt
        return yt, epsilon, std, self.g(t, yt)

    def sample_debiasing_t(self, shape):
        """uniform t (the likelihood weighting g^2 / std^2 of the VE-SDE is constant in t)"""
        return self.t_epsilon + torch.rand(*shape) * (self.T - self.t_epsilon)

    def sample_t_device(self, shape, device, debias=True, eps=1e-4):
        """`sample_t` of the models (models/diffusion.py: `sample_debiasing_t` + eps, folded back where it exceeds T; or
        eps + u T without debiasing) drawn on `device` from the CUDA generator: an affine map of one torch.rand, no host
        work, so a CUDA-graph capture of the training step can contain it."""
        u = torch.rand(*shape, device=device, dtype=torch.float32)
        if debias:
            t = self.t_epsilon + u * (self.T - self.t_epsilon) + eps
            return torch.where(t > self.T, t - eps, t)
        t = eps + u * self.T
        return torch.where(t > self.T, torch.full_like(t, self.T - eps), t)


class PluginReverseSDE(torch.nn.Module):
    """Reverse-time SDE with plug-in drift a = g * score:  mu = g a - f,  sigma = g  (time runs T - t)."""

    def __init__(self, base_sde, drift_a, T, vtype='rademacher', debias=False):
        super().__init__()
        self.base_sde = base_sde
        self.a = drift_a
        self.T = T
        self.vtype = vtype
        self.debias = debias

    def mu(self, t, x, cond, lmbd=0.):
        s = self.T - t
        return (1. - 0.5 * lmbd) * self.base_sde.g(s, x) * self.a(x, cond, s) - self.base_sde.f(s, x)

    def sigma(self, t, y, lmbd=0.):
        return (1. - lmbd) ** 0.5 * self.base_sde.g(self.T - t, y)
