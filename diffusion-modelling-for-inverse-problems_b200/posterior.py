"""PosteriorLoss (DPS joint loss, losses.py:340-386) as one fused forward+backward call (`dmip_posterior_loss_fwd_bwd`):
prior-net pass with xdim tangent streams (DSM + J_s), surrogate VJP at the Tweedie mean, target assembly, likelihood-net
pass — parameter gradients of both nets come back in flat buffers handed to autograd."""
import ctypes as C

import torch

from . import _lib


class DmipPosteriorLoss(C.Structure):
    _fields_ = [("xdim", C.c_int32), ("ydim", C.c_int32), ("batch", C.c_int64), ("batch_global", C.c_int64),
                ("prior_net", _lib.DmipMlp), ("lik_net", _lib.DmipMlp), ("surrogate", _lib.DmipMlp),
                ("beta_min", C.c_float), ("beta_max", C.c_float), ("a", C.c_float), ("b", C.c_float), ("lam", C.c_float),
                ("x", C.c_void_p), ("y", C.c_void_p), ("t", C.c_void_p), ("eps", C.c_void_p),
                ("out_losses", C.c_void_p), ("grad_prior", C.c_void_p), ("grad_lik", C.c_void_p),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
                ("sde_kind", C.c_int32), ("sigma_min", C.c_float), ("sigma_max", C.c_float)]


def _bind():
    L = _lib.require_gpu()
    if not getattr(L, "_post_bound", False):
        L.dmip_posterior_loss_workspace_bytes.restype = C.c_size_t
        L.dmip_posterior_loss_workspace_bytes.argtypes = [C.POINTER(DmipPosteriorLoss)]
        L.dmip_posterior_loss_fwd_bwd.restype = C.c_int
        L.dmip_posterior_loss_fwd_bwd.argtypes = [C.POINTER(DmipPosteriorLoss), C.c_void_p]
        L.dmip_loss_grad_floats.restype = C.c_size_t
        L.dmip_loss_grad_floats.argtypes = [C.POINTER(_lib.DmipMlp)]
        L._post_bound = True
    return L


class _FusedPosteriorLoss(torch.autograd.Function):

    @staticmethod
    def forward(ctx, cfg, x, y, t, eps, *params):
        L = _bind()
        dev = x.device
        keep = []
        d = DmipPosteriorLoss()
        d.xdim, d.ydim = x.shape[1], y.shape[1]
        d.batch = x.shape[0]
        d.batch_global = cfg.get('batch_global', 0) or x.shape[0]
        d.prior_net = _lib.mlp_desc(cfg['prior_net'], keep)
        d.lik_net = _lib.mlp_desc(cfg['lik_net'], keep)
        d.surrogate = _lib.mlp_desc(cfg['forward_model'], keep)
        _lib.set_sde(d, cfg['base_sde'])
        d.a, d.b, d.lam = cfg['a'], cfg['b'], cfg['lam']
        for name, v in (('x', x), ('y', y), ('t', t.reshape(-1)), ('eps', eps)):
            v = v.detach().to(dev, torch.float32).contiguous()
            keep.append(v)
            setattr(d, name, v.data_ptr())
        losses = torch.empty(4, device=dev, dtype=torch.float32)
        n1 = L.dmip_loss_grad_floats(C.byref(d.prior_net))
        n2 = L.dmip_loss_grad_floats(C.byref(d.lik_net))
        go = cfg.get('grad_out')     # data-parallel step: one flat bucket [prior | likelihood] (dmip.distributed.GradBucket)
        if go is not None:
            assert go.is_cuda and go.dtype == torch.float32 and go.is_contiguous() and go.numel() == n1 + n2
            g1, g2 = go[:n1], go[n1:]
        else:
            g1 = torch.empty(n1, device=dev, dtype=torch.float32)
            g2 = torch.empty(n2, device=dev, dtype=torch.float32)
        d.out_losses, d.grad_prior, d.grad_lik = losses.data_ptr(), g1.data_ptr(), g2.data_ptr()
        nbytes = L.dmip_posterior_loss_workspace_bytes(C.byref(d))
        if nbytes == 0:
            _lib.check(-1)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        d.workspace, d.workspace_bytes = ws.data_ptr(), nbytes
        with torch.cuda.device(dev):
            _lib.check(L.dmip_posterior_loss_fwd_bwd(C.byref(d), _lib.stream_ptr()))
        cfg['launches'] = L.dmip_last_launch_count()
        ctx.flats = (g1, g2)
        ctx.shapes = cfg['shapes']
        return losses

    @staticmethod
    def backward(ctx, gout):
        scale = gout[0]
        grads = []
        for flat, shapes in zip(ctx.flats, ctx.shapes):
            off = 0
            for shp in shapes:
                n = shp.numel()
                grads.append((flat[off:off + n] * scale).view(shp))
                off += n
        return (None, None, None, None, None, *grads)


class _NoCtx:
    """stand-in for the autograd context when the kernel is called without an autograd edge"""


def posterior_loss_fused(loss_mod, model, x, y, t, eps=None):
    """loss_mod: PosteriorLoss; model: PluginReverseSDE whose drift `a` is a PosteriorScore.  `eps` (optional) injects
    the forward-SDE draw that `base_sde.sample` would make (losses.py:374)."""
    if not x.is_cuda:
        raise RuntimeError("dmip fused losses run on CUDA (sm_100a) only: there is no CPU fallback")
    prior, lik = model.a.prior_net, model.a.likelihood_net
    if eps is None:
        eps = torch.randn_like(x)
    p1 = [p for lin in _lib.linear_layers(prior) for p in (lin.weight, lin.bias)]
    p2 = [p for lin in _lib.linear_layers(lik) for p in (lin.weight, lin.bias)]
    cfg = dict(prior_net=prior, lik_net=lik, forward_model=loss_mod.forward_model,
               base_sde=model.base_sde,
               a=float(loss_mod.a), b=float(loss_mod.b), lam=float(loss_mod.lam),
               batch_global=getattr(loss_mod, 'batch_global', 0), grad_out=getattr(loss_mod, 'grad_out', None),
               shapes=([p.shape for p in p1], [p.shape for p in p2]))
    if cfg['grad_out'] is not None:      # raw mode: no autograd edge, the gradients land in the caller's bucket
        out = _FusedPosteriorLoss.forward(_NoCtx(), cfg, x, y, t, eps, *p1, *p2)
    else:
        out = _FusedPosteriorLoss.apply(cfg, x, y, t, eps, *p1, *p2)
    loss_mod.last_launch_count = cfg['launches']
    return out[0], {'PriorLoss': out[1].detach(), 'LikelihoodLoss': out[2].detach()}
