"""Drop-in for the reference's `losses.py`: DSMLoss, ScoreFPELoss, ConditionalScoreFPELoss, DSM_PDELoss, PINNLoss,
PINNLoss2, PosteriorLoss — same class names, constructor arguments, `.name` dispatch keys and `forward` signatures.

The reference builds these losses out of 2d+1 `torch.autograd.grad(create_graph=True)` passes and then runs
`loss.backward()` through the double-backward graph (losses.py:14-26, 77-98, 214-242).  Here the composite losses
(PINNLoss, DSM_PDELoss, the DSM branch of `train_epoch`, PosteriorLoss) are single fused forward+backward calls into
libdmip_sm100.so (`dmip_loss_fwd_bwd`, include/dmip.h): forward-mode jets give the exact divergence, the total
time derivative and grad_x in one sweep, and the parameter gradients come back in a flat buffer that a
`torch.autograd.Function` hands to `loss.backward()`, so the usual
`optimizer.zero_grad(); loss.backward(); optimizer.step()` of the reference's train loop is unchanged.

The forward SDE is the model's `base_sde`: the reference's VariancePreservingSDE or sdes.VarianceExplodingSDE (same
kernels; the score is a / g for both, and the VE Score-FPE residual is ds/dt - g^2/2 grad_x [div s + |s|^2], f = 0).

Numerical contract (SURVEY.md Q8-Q10): ds/dt is the total derivative along x_t(t) at fixed noise; grad_x is a
constant in the backward pass; the (B,)+(B,1) broadcast of the reference is reproduced as the value it evaluates to,
mean(dsm)+mean(ic)+mean(pde), without materialising the (B,B) matrix.
"""
import ctypes as C

import torch
from torch import nn

from . import _lib

_LOSS_DSM, _LOSS_DSM_PDE, _LOSS_PINN, _LOSS_PINN2 = 0, 1, 2, 3
_METRIC = {'L1': 1, 'L2': 2}
_DIVERGENCE = {'exact': 0, 'hutchinson': 1, 'approx': 1, 'approximate': 1, 'exact_adjoint': 2}


def rademacher_like(s):
    """+-1 with probability 1/2 each (losses.py:7-11), drawn on the device of `s`."""
    return torch.randint(0, 2, s.shape, device=s.device).to(s.dtype) * 2 - 1


def _divergence(loss_fn, z):
    """divergence_method of ScoreFPELoss.forward (losses.py:81-86) -> (code, probe or None).  The probe of the
    Hutchinson estimator is drawn like div_estimator does (one Rademacher sample) unless `loss_fn.probe` injects one."""
    m = getattr(loss_fn, 'divergence_method', 'exact')
    if m not in _DIVERGENCE:
        raise ValueError('No valid value for divergence method specified. Need to be one of "exact","hutchinson",'
                         '"approx" or "approximate", but {} was given'.format(m))
    code = _DIVERGENCE[m]
    if code != 1 or loss_fn.pde_loss.name != 'FPELoss':
        return code, None
    v = getattr(loss_fn, 'probe', None)
    return code, (rademacher_like(z) if v is None else v)


class DmipLoss(C.Structure):
    _fields_ = [("kind", C.c_int32), ("model", C.c_int32), ("xdim", C.c_int32), ("ydim", C.c_int32),
                ("batch", C.c_int64), ("batch_global", C.c_int64), ("net", _lib.DmipMlp),
                ("beta_min", C.c_float), ("beta_max", C.c_float), ("lam", C.c_float), ("lam2", C.c_float),
                ("pde_loss", C.c_int32), ("pde_metric", C.c_int32), ("ic_metric", C.c_int32), ("divergence", C.c_int32),
                ("x", C.c_void_p), ("y", C.c_void_p), ("t", C.c_void_p), ("eps", C.c_void_p),
                ("ic_target", C.c_void_p), ("hutch_v", C.c_void_p), ("out_losses", C.c_void_p), ("grad", C.c_void_p),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
                ("sde_kind", C.c_int32), ("sigma_min", C.c_float), ("sigma_max", C.c_float)]


def _bind():
    L = _lib.require_gpu()
    if not getattr(L, "_loss_bound", False):
        L.dmip_loss_workspace_bytes.restype = C.c_size_t
        L.dmip_loss_workspace_bytes.argtypes = [C.POINTER(DmipLoss)]
        L.dmip_loss_grad_floats.restype = C.c_size_t
        L.dmip_loss_grad_floats.argtypes = [C.POINTER(_lib.DmipMlp)]
        L.dmip_loss_fwd_bwd.restype = C.c_int
        L.dmip_loss_fwd_bwd.argtypes = [C.POINTER(DmipLoss), C.c_void_p]
        L._loss_bound = True
    return L


def _metric(m):
    if m not in _METRIC:
        raise ValueError('No valid metric specified. Metric should be one of "L1" or "L2" but was {}'.format(m))
    return _METRIC[m]


def _launch_fused(net, cfg, x, y, t, eps, ic_target, grad_out=None):
    """One dmip_loss_fwd_bwd call.  Returns (losses[4], flat gradient, kernel launches).  `grad_out`: a caller-owned flat
    fp32 buffer (dmip_loss_grad_floats(net) elements) the kernels write the gradient into — the data-parallel step hands
    in its all-reduce bucket, whose slices ARE the parameters' .grad (dmip.distributed.GradBucket)."""
    L = _bind()
    dev = x.device
    d = DmipLoss()
    d.kind, d.model = cfg['kind'], cfg['model']
    d.xdim, d.ydim = x.shape[1], y.shape[1]
    d.batch = x.shape[0]
    d.batch_global = cfg.get('batch_global', 0) or x.shape[0]
    d.net, keep = _lib.mlp_desc_cached(net)
    _lib.set_sde(d, cfg['base_sde'])
    d.lam, d.lam2 = cfg.get('lam', 0.0), cfg.get('lam2', 0.0)
    d.pde_loss, d.pde_metric, d.ic_metric = cfg.get('pde_loss', 0), cfg.get('pde_metric', 1), cfg.get('ic_metric', 1)
    d.divergence = cfg.get('divergence', 0)
    tens = {}
    for name, v in (('x', x), ('y', y), ('t', t.reshape(-1)), ('eps', eps), ('ic_target', ic_target),
                    ('hutch_v', cfg.get('hutch_v'))):
        if v is None:
            continue
        v = v.detach().to(dev, torch.float32).contiguous()
        tens[name] = v
        setattr(d, name, v.data_ptr())
    guard = _lib.Guarded()
    losses = guard.empty(4, torch.float32, dev)
    n_grad = L.dmip_loss_grad_floats(C.byref(d.net))
    if grad_out is None:
        grad = guard.empty(n_grad, torch.float32, dev)
    else:
        grad = grad_out
        assert grad.is_cuda and grad.dtype == torch.float32 and grad.is_contiguous() and grad.numel() == n_grad
    d.out_losses, d.grad = losses.data_ptr(), grad.data_ptr()
    nbytes = L.dmip_loss_workspace_bytes(C.byref(d))
    if nbytes == 0:
        _lib.check(-1)
    ws = guard.empty(nbytes, torch.uint8, dev)
    d.workspace, d.workspace_bytes = ws.data_ptr(), nbytes
    if torch.cuda.current_device() == dev.index:
        _lib.check(L.dmip_loss_fwd_bwd(C.byref(d), _lib.stream_ptr()))
    else:
        with torch.cuda.device(dev):
            _lib.check(L.dmip_loss_fwd_bwd(C.byref(d), _lib.stream_ptr()))
    guard.check("dmip_loss_fwd_bwd")
    return losses, grad, L.dmip_last_launch_count()


class _FusedLoss(torch.autograd.Function):
    """forward: one dmip_loss_fwd_bwd call -> losses[4]; backward: hands the flat gradient to the parameters."""

    @staticmethod
    def forward(ctx, net, cfg, x, y, t, eps, ic_target, *params):
        losses, grad, cfg['launches'] = _launch_fused(net, cfg, x, y, t, eps, ic_target)
        ctx.flat = grad
        ctx.shapes = [p.shape for p in params]
        return losses

    @staticmethod
    def backward(ctx, gout):
        # only losses[0] (the total) is differentiable; the rest is the info dict.  ONE multiply over the flat gradient;
        # the parameters get views of the product (AccumulateGrad adopts them when .grad is None: no copies)
        flat = ctx.flat * gout[0]
        grads, off = [], 0
        for shp in ctx.shapes:
            n = shp.numel()
            grads.append(flat[off:off + n].view(shp))
            off += n
        return (None, None, None, None, None, None, None, *grads)


def _fused(sde, cfg, x, y, t, eps, ic_target=None):
    """Run the fused kernel for the net `sde.a`; returns the tensor losses[4] whose [0] carries the autograd edge."""
    net = sde.a
    if not x.is_cuda:
        raise RuntimeError("dmip fused losses run on CUDA (sm_100a) only: there is no CPU fallback")
    cfg = dict(cfg, base_sde=sde.base_sde)
    grad_out = cfg.pop('grad_out', None)
    if grad_out is not None:                  # raw mode (data-parallel step): no autograd edge, gradient lands in grad_out
        out, _, cfg['launches'] = _launch_fused(net, cfg, x, y, t, eps, ic_target, grad_out)
        return out, cfg
    params = [p for lin in _lib.linear_layers(net) for p in (lin.weight, lin.bias)]
    return _FusedLoss.apply(net, cfg, x, y, t, eps, ic_target, *params), cfg


def _check_diffused(model, x, y, diffused_samples, t, target, std):
    """The fused kernels re-derive x_t = alpha(t) z_0 + std(t) eps from (x, y, t, eps) in-kernel.  A caller that hands in the
    reference's full argument list (std is a tensor) gets it validated: a different x_t would silently give a different
    loss than the reference.  The internal train loop passes std=None and skips this (no host sync on the hot path)."""
    if std is None or not torch.is_tensor(diffused_samples):
        return
    z0 = x if diffused_samples.shape[1] == x.shape[1] else torch.cat([x, y], dim=1)
    tt = t.detach().reshape(-1, 1)
    want = model.base_sde.mean_weight(tt) * z0 + model.base_sde.var(tt) ** 0.5 * target
    if not torch.allclose(diffused_samples.detach(), want, rtol=1e-4, atol=1e-5):
        raise ValueError("diffused_samples is not alpha(t) * [x(,y)] + std(t) * target: the fused loss kernels re-derive "
                         "x_t from (x, y, t, target) and cannot take an arbitrary x_t (INTEGRATION.md, deviations)")


class DSMLoss(nn.Module):
    """Denoising score matching, per sample: 1/2 * sum_d (s*std + eps)^2."""

    def __init__(self):
        super().__init__()
        self.name = 'DSMLoss'

    def forward(self, s, std, target):
        return ((s * std + target) ** 2).view(s.shape[0], -1).sum(1, keepdim=False) / 2


class ScoreFPELoss(nn.Module):
    """Residual of the score Fokker–Planck equation  d_t s = beta/2 grad_x (div_x s + |s|^2 + x.s)  (VE-SDE:
    d_t s = g^2/2 grad_x (div_x s + |s|^2)).
    Carries `name` / `metric`; its evaluation is fused into PINNLoss / DSM_PDELoss (forward-mode jets through the
    net need the net, not a detached score tensor)."""

    def __init__(self, metric='L1'):
        super().__init__()
        self.name = 'FPELoss'
        self.metric = metric

    def forward(self, s, x_t, t, beta, divergence_method='exact'):
        raise RuntimeError("ScoreFPELoss is evaluated inside the fused PINNLoss / DSM_PDELoss kernels "
                           "(dmip_loss_fwd_bwd); call those with the model instead of a score tensor")


class ConditionalScoreFPELoss(nn.Module):
    """cScoreFPE: sum_d (std^3 ds/dt - eps beta alpha^2 / 2)^2 (L2) or abs (L1); fused like ScoreFPELoss."""

    def __init__(self, metric='L2'):
        super().__init__()
        self.name = 'cScoreFPELoss'
        self.metric = metric

    def forward(self, s, t, alpha, beta, target, std):
        raise RuntimeError("ConditionalScoreFPELoss is evaluated inside the fused PINNLoss / DSM_PDELoss kernels")


def _model_kind(x, diffused_samples):
    return _lib.CDE if diffused_samples.shape[1] == x.shape[1] else _lib.CDIFFE


class DSM_PDELoss(nn.Module):
    """DSM + lam * PDE residual (Lai et al. 2023)."""

    def __init__(self, lam=1., pde_loss='FPE', pde_metric='L1', *, divergence_method='exact'):
        super().__init__()
        self.lam = lam
        self.dsm_loss = DSMLoss()
        self.pde_loss = ScoreFPELoss(pde_metric) if pde_loss == 'FPE' else ConditionalScoreFPELoss(pde_metric)
        self.name = 'DSM_PDELoss'
        self.divergence_method = divergence_method

    def forward(self, model, x, y, diffused_samples, t, target, std, g):
        div, probe = _divergence(self, diffused_samples)
        _check_diffused(model, x, y, diffused_samples, t, target, std)
        cfg = dict(kind=_LOSS_DSM_PDE, model=_model_kind(x, diffused_samples), lam=float(self.lam),
                   pde_loss=0 if self.pde_loss.name == 'FPELoss' else 1, pde_metric=_metric(self.pde_loss.metric),
                   divergence=div, hutch_v=probe, batch_global=getattr(self, 'batch_global', 0),
                   grad_out=getattr(self, 'grad_out', None))
        out, cfg = _fused(model, cfg, x, y, t, target)
        self.last_launch_count = cfg['launches']
        return out[0], {'PDE-Loss': out[3].detach(), 'DSM-Loss': out[1].detach()}


class PINNLoss(nn.Module):
    """DSM + lam2 * initial condition at t=0 + lam * PDE residual (Raissi et al. 2019 style)."""

    def __init__(self, initial_condition, lam=1., lam2=1., pde_loss='FPE', ic_metric='L1', pde_metric='L1', *,
                 divergence_method='exact'):
        super().__init__()
        self.divergence_method = divergence_method
        self.lam = lam
        self.lam2 = lam2
        self.initial_condition = initial_condition
        self.pde_loss = ConditionalScoreFPELoss(pde_metric) if pde_loss == 'cScoreFPE' else ScoreFPELoss(pde_metric)
        self.dsm_loss = DSMLoss()
        self.name = 'PINNLoss'
        self.ic_metric = ic_metric

    def forward(self, model, x, y, diffused_samples, t, target, std, g):
        div, probe = _divergence(self, diffused_samples)
        cfg = dict(kind=_LOSS_PINN, model=_model_kind(x, diffused_samples), lam=float(self.lam), lam2=float(self.lam2),
                   pde_loss=0 if self.pde_loss.name == 'FPELoss' else 1, pde_metric=_metric(self.pde_loss.metric),
                   ic_metric=_metric(self.ic_metric), divergence=div, hutch_v=probe,
                   batch_global=getattr(self, 'batch_global', 0), grad_out=getattr(self, 'grad_out', None))
        _check_diffused(model, x, y, diffused_samples, t, target, std)
        with torch.no_grad():
            ic_target = self.initial_condition(x, y)
        out, cfg = _fused(model, cfg, x, y, t, target, ic_target)
        self.last_launch_count = cfg['launches']
        return out[0], {'PDE-Loss': out[3].detach(), 'Initial Condition': out[2].detach(), 'DSM-Loss': out[1].detach()}


class PINNLoss2(nn.Module):
    """PINNLoss without the data-driven DSM term: mean(lam2 * initial condition + lam * PDE residual); the DSM loss is only
    reported ('DSM_eval').  Constructor as upstream (losses.py:250-261) — so `utils.get_model_from_args`, which passes an
    unsupported `pde_metric=` (utils.py:38), fails with the same TypeError — plus the attribute upstream's forward reads
    but never sets (`ic_metric`, losses.py:276), as a keyword-only argument (default 'L1', PINNLoss's default).  The pde
    losses keep their default metrics (ScoreFPELoss 'L1', ConditionalScoreFPELoss 'L2')."""

    def __init__(self, initial_condition, lam=1., lam2=1., pde_loss='FPE', *, ic_metric='L1', divergence_method='exact'):
        super().__init__()
        self.lam = lam
        self.lam2 = lam2
        self.initial_condition = initial_condition
        self.pde_loss = ScoreFPELoss() if pde_loss == 'FPE' else ConditionalScoreFPELoss()
        self.eval_metric = DSMLoss()
        self.name = 'PINNLoss2'
        self.ic_metric = ic_metric
        self.divergence_method = divergence_method

    def forward(self, model, x, y, diffused_samples, t, target, std, g):
        div, probe = _divergence(self, diffused_samples)
        cfg = dict(kind=_LOSS_PINN2, model=_model_kind(x, diffused_samples), lam=float(self.lam), lam2=float(self.lam2),
                   pde_loss=0 if self.pde_loss.name == 'FPELoss' else 1, pde_metric=_metric(self.pde_loss.metric),
                   ic_metric=_metric(self.ic_metric), divergence=div, hutch_v=probe,
                   batch_global=getattr(self, 'batch_global', 0), grad_out=getattr(self, 'grad_out', None))
        _check_diffused(model, x, y, diffused_samples, t, target, std)
        with torch.no_grad():
            ic_target = self.initial_condition(x, y)
        out, cfg = _fused(model, cfg, x, y, t, target, ic_target)
        self.last_launch_count = cfg['launches']
        return out[0], {'PDE-Loss': out[3].detach(), 'Initial Condition': out[2].detach(), 'DSM_eval': out[1].detach()}


class PosteriorLoss(nn.Module):
    """Joint loss of the DPS prior / likelihood nets (Chung et al. 2023 with learned scores); scatterometry only,
    as upstream."""

    def __init__(self, forward_model, a, b, lam):
        super().__init__()
        self.name = 'PosteriorLoss'
        self.dsm_loss = DSMLoss()
        self.forward_model = forward_model
        self.a = a
        self.b = b
        self.lam = lam

    def forward(self, model, x, y, t, eps=None):
        from .posterior import posterior_loss_fused
        return posterior_loss_fused(self, model, x, y, t, eps)


def dsm_fused(model, x, y, t, eps, batch_global=0, grad_out=None):
    """mean_B DSMLoss(a(x_t, y, t)/g, std, eps) with its parameter gradient — the `loss_fn.name == 'DSMLoss'` branch of
    CDE/CDiffE.train_epoch (models/diffusion.py:83-85, :134-137) as one fused call.  Returns (loss, launches)."""
    cfg = dict(kind=_LOSS_DSM, model=_lib.CDE if model.variant == 'CDE' else _lib.CDIFFE, batch_global=batch_global,
               grad_out=grad_out)
    out, cfg = _fused(model.sde, cfg, x, y, t, eps)
    return out[0], cfg['launches']


def fused_train_step(model, loss_fn, x, y, t):
    """Body of the reference's train_epoch loops (models/diffusion.py:80-88, :129-139, :211) for one batch:
    draw the forward-SDE noise, evaluate the loss with the fused kernels, return (loss, info)."""
    if loss_fn.name == 'PosteriorLoss':
        return loss_fn(model.sde, x, y, t)
    z = x if model.variant == 'CDE' else torch.cat([x, y], dim=1)
    eps = torch.randn_like(z)                                   # VariancePreservingSDE.sample's draw (sdes.py:45)
    if loss_fn.name == 'DSMLoss':
        loss, loss_fn.last_launch_count = dsm_fused(model, x, y, t, eps, getattr(loss_fn, 'batch_global', 0),
                                                    getattr(loss_fn, 'grad_out', None))
        return loss, {}
    # composite losses take the reference's argument list; the diffused samples are re-derived in-kernel from
    # (x, y, t, eps), so only their width (CDE vs CDiffE) is read from the tensor passed here
    return loss_fn(model.sde, x, y, z, t, eps, None, None)
