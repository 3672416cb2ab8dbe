"""Score-training losses under the VE-SDE — fp64 restatement of oracle/losses.py with the variance-exploding forward
process (TEST INFRASTRUCTURE ONLY; oracle/losses.py, which the golden fixtures pin, is the VP oracle and stays as it is).

PARITY UNPINNED: upstream trains only on the VP-SDE.  This module is what the fused kernels' VE path is checked
against, and `tests/test_ve_loss_oracle.py` pins it to a literal autograd statement and to the PDE itself.

    sigma(t) = smin (smax / smin)^t,  lr = ln(smax / smin),  f = 0,  g^2 = 2 lr sigma^2,  alpha = 1,  var = sigma^2
    x_t = z0 + sigma eps,  dx_t/dt = eps sigma lr,  s = a / g  (the plug-in convention of the samplers)
    ds/dt  = a_dot / g - a lr / g                         (total derivative along x_t(t) at fixed eps, fact Q8)
    Score-FPE residual  R = ds/dt - g^2/2 grad_x [div s + |s|^2]   (no x.s term: f = 0), grad_x detached (Q9)
        grad_x [div s + |s|^2] = gtr / g + 2 J^T a / g^2
    cScoreFPE  r = std^3 ds/dt - eps g^2 / 2
    PINN initial condition  s(x, y, 0) = a / g(0),  g(0) = smin sqrt(2 lr)
    PosteriorLoss  x0_hat = x_t + sigma^2 s_prior,  target = (sigma^2 J_s^T + I) u,  lik = sum (s_lik - target)^2
"""
import math

import torch

from . import nets as onets
from . import scatterometry as scat
from .losses import dsm

SIGMA_MIN = 0.01          # sdes.VarianceExplodingSDE defaults
SIGMA_MAX = 50.0


class VESDE:
    def __init__(self, sigma_min=SIGMA_MIN, sigma_max=SIGMA_MAX):
        self.smin, self.smax = float(sigma_min), float(sigma_max)
        self.lr = math.log(self.smax / self.smin)

    def sigma(self, t):
        return self.smin * torch.exp(t * self.lr)

    def g2(self, t):
        return 2.0 * self.lr * self.sigma(t) ** 2

    def perturb(self, t, z0, eps):
        """x_t = z0 + sigma(t) eps -> (x_t, std)"""
        std = self.sigma(t)
        return z0 + std * eps, std

    def xdot(self, t, eps):
        """d/dt x_t at fixed eps"""
        return eps * self.sigma(t) * self.lr


def ds_dt(sde, a, a_dot, t):
    """d(a / g)/dt from the tangent a_dot of the net output: a_dot / g - a lr / g"""
    g = sde.g2(t) ** 0.5
    return a_dot / g - a * sde.lr / g


def grad_phi(a, J, gtr, g2):
    """grad_x [div s + |s|^2] with s = a / g (g constant in x): gtr / g + 2 J^T a / g^2; J[b,i,k] = d a_i / d x_k,
    gtr[b,k] = grad_x of tr J (or of the Hutchinson estimate) at x"""
    return gtr / g2 ** 0.5 + 2 * torch.einsum("bik,bi->bk", J, a) / g2


def fpe_residual(ds_dt_, g2, grad_x):
    return ds_dt_ - 0.5 * g2 * grad_x


def score_and_fpe_terms(sde, params, z_t, cond, t, eps, need_space=True, probe=None):
    """oracle/losses.py score_and_fpe_terms under the VE-SDE (same jets, same probe convention)."""
    B, d = z_t.shape
    c = 0 if cond is None else cond.shape[1]
    inp = torch.cat([z_t] + ([cond] if c else []) + [t.reshape(B, 1)], dim=1)
    nin = inp.shape[1]
    zeros = torch.zeros(B, nin, dtype=inp.dtype)
    dirs = [torch.cat([sde.xdot(t, eps), torch.zeros(B, c, dtype=inp.dtype), torch.ones(B, 1, dtype=inp.dtype)], 1)]
    pairs = []
    if need_space:
        for k in range(d):
            e = zeros.clone()
            e[:, k] = 1.0
            dirs.append(e)
        if probe is None:
            pairs = [(1 + i, 1 + k) for i in range(d) for k in range(i, d)]
        else:
            dirs.append(torch.cat([probe, torch.zeros(B, nin - d, dtype=inp.dtype)], 1))
            pairs = [(d + 1, 1 + k) for k in range(d)]
    a, ad, add = onets.mlp_jets(params, inp, dirs, pairs)
    g2 = sde.g2(t)
    g = g2 ** 0.5
    out = {"a": a, "s": a / g, "g2": g2, "ds_dt": ds_dt(sde, a, ad[0], t)}
    if need_space:
        J = torch.stack(ad[1:1 + d], dim=2)
        gtr = torch.zeros(B, d, dtype=inp.dtype)
        if probe is None:
            out["div_s"] = torch.diagonal(J, dim1=1, dim2=2).sum(1, keepdim=True) / g
            for idx, (i, k) in enumerate(pairs):
                i -= 1
                k -= 1
                gtr[:, k] += add[idx][:, i]
                if i != k:
                    gtr[:, i] += add[idx][:, k]
        else:
            out["div_s"] = (probe * ad[1 + d]).sum(1, keepdim=True) / g
            for k in range(d):
                gtr[:, k] = (probe * add[k]).sum(1)
        out["grad_x"] = grad_phi(a, J, gtr, g2).detach()
    return out


def score_fpe(terms, metric="L1"):
    R = fpe_residual(terms["ds_dt"], terms["g2"], terms["grad_x"])
    if metric == "L1":
        return R.abs().mean(1, keepdim=True)
    if metric == "L2":
        return (R ** 2).mean(1, keepdim=True)
    raise ValueError(metric)


def cscore_residual(terms, eps, std):
    return std ** 3 * terms["ds_dt"] - 0.5 * eps * terms["g2"]


def cscore_fpe(terms, eps, std, metric="L2"):
    r = cscore_residual(terms, eps, std)
    return (r ** 2).sum(1) if metric == "L2" else r.abs().sum(1)


def _pde(terms, eps, std, pde_loss, pde_metric):
    if pde_loss == "cScoreFPE":
        return cscore_fpe(terms, eps, std, pde_metric)
    return score_fpe(terms, pde_metric)


def split(sde, model_kind, x, y, t, eps):
    if model_kind == "CDE":
        z0, cond = x, y
    elif model_kind == "CDiffE":
        z0, cond = torch.cat([x, y], 1), None
    else:
        raise ValueError(model_kind)
    z_t, std = sde.perturb(t, z0, eps)
    return z0, cond, z_t, std


def initial_score(sde, params, x, y):
    """s(x, y, 0) = a(x, y, 0) / g(0)"""
    t0 = torch.zeros(x.shape[0], 1, dtype=x.dtype)
    return onets.mlp(params, x, y, t0) / sde.g2(t0) ** 0.5


def dsm_loss(sde, params, model_kind, x, y, t, eps):
    z0, cond, z_t, std = split(sde, model_kind, x, y, t, eps)
    a = onets.mlp(params, z_t, cond, t)
    return dsm(a / sde.g2(t) ** 0.5, std, eps).mean()


def dsm_pde_loss(sde, params, model_kind, x, y, t, eps, lam=1.0, pde_loss="FPE", pde_metric="L1", probe=None):
    z0, cond, z_t, std = split(sde, model_kind, x, y, t, eps)
    terms = score_and_fpe_terms(sde, params, z_t, cond, t, eps, need_space=(pde_loss != "cScoreFPE"), probe=probe)
    l_dsm = dsm(terms["s"], std, eps)
    l_pde = lam * _pde(terms, eps, std, pde_loss, pde_metric)
    return l_dsm.mean() + l_pde.mean(), {"PDE-Loss": l_pde.mean(), "DSM-Loss": l_dsm.mean()}


def pinn_loss(sde, params, model_kind, x, y, t, eps, ic_target, lam=1.0, lam2=1.0,
              pde_loss="FPE", ic_metric="L1", pde_metric="L1", probe=None):
    xdim = x.shape[1]
    z0, cond, z_t, std = split(sde, model_kind, x, y, t, eps)
    s0 = initial_score(sde, params, x, y)
    terms = score_and_fpe_terms(sde, params, z_t, cond, t, eps, need_space=(pde_loss != "cScoreFPE"), probe=probe)
    diff = s0[:, :xdim] - ic_target
    l_ic = lam2 * ((diff ** 2).mean(1, keepdim=True) if ic_metric == "L2" else diff.abs().mean(1, keepdim=True))
    l_dsm = dsm(terms["s"], std, eps)
    l_pde = lam * _pde(terms, eps, std, pde_loss, pde_metric)
    loss = l_dsm.mean() + l_ic.mean() + l_pde.mean()
    return loss, {"PDE-Loss": l_pde.mean(), "Initial Condition": l_ic.mean(), "DSM-Loss": l_dsm.mean()}


def pinn2_loss(sde, params, model_kind, x, y, t, eps, ic_target, lam=1.0, lam2=1.0,
               pde_loss="FPE", ic_metric="L1", probe=None):
    xdim = x.shape[1]
    z0, cond, z_t, std = split(sde, model_kind, x, y, t, eps)
    s0 = initial_score(sde, params, x, y)
    terms = score_and_fpe_terms(sde, params, z_t, cond, t, eps, need_space=(pde_loss != "cScoreFPE"), probe=probe)
    diff = s0[:, :xdim] - ic_target
    l_ic = lam2 * ((diff ** 2).mean(1, keepdim=True) if ic_metric == "L2" else diff.abs().mean(1, keepdim=True))
    l_pde = lam * _pde(terms, eps, std, pde_loss, "L2" if pde_loss == "cScoreFPE" else "L1")
    return l_ic.mean() + l_pde.mean(), {"PDE-Loss": l_pde.mean(), "Initial Condition": l_ic.mean(),
                                        "DSM_eval": dsm(terms["s"], std, eps).mean()}


def posterior_loss(sde, prior_params, lik_params, surr_params, x, y, t, eps, lam, a=scat.A_NOISE, b=scat.B_NOISE):
    """oracle/losses.py posterior_loss under the VE-SDE (alpha = 1, std = sigma(t))"""
    x_t, std = sde.perturb(t, x, eps)
    x_t = x_t.detach().requires_grad_(True)
    s_prior = onets.mlp2(prior_params, x_t, t)
    s_lik = onets.mlp(lik_params, x_t, y, t)
    l_prior = dsm(s_prior, std, eps)
    x0_hat = (x_t + std ** 2 * s_prior).detach()
    fx = scat.surrogate(surr_params, x0_hat)
    pre = (a * fx) ** 2 + b ** 2
    w = -a * a * fx / pre + (y - fx) / pre + a * a * (y - fx) ** 2 * fx / pre
    u = scat.surrogate_vjp(surr_params, x0_hat, w)
    vhp = torch.autograd.grad(s_prior, x_t, u, retain_graph=True)[0]
    target = (std ** 2 * vhp + u).detach()
    l_lik = ((s_lik - target) ** 2).sum(1)
    loss = (l_prior + lam * l_lik).mean()
    return loss, {"PriorLoss": l_prior.mean(), "LikelihoodLoss": lam * l_lik.mean()}
