"""Drop-in for the reference's `nets.py` score networks (MLP :17-35, MLP2 :37-57, PosteriorScore :143-157).

The modules keep the reference's parameter layout — `state_dict()` keys `0,3,5,7.{weight,bias}` (SURVEY.md Q2) —
and its numerics: tanh is applied twice after the first Linear, because the reference registers its activation a
second time under the name 'act' and `nn.Sequential.forward` walks every registered module (SURVEY.md Q1).  That is
reproduced here on purpose so reference checkpoints (`current_model.pt`, `diffusion.pt`) load and behave identically.

`forward` on CUDA tensors without autograd runs the fused kernels of libdmip_sm100.so (`dmip_mlp_forward`); when
autograd is recording it runs `dmip_mlp_forward_stash` and registers `dmip_mlp_backward` as its backward (tcgen05 kernels:
parameter and input gradients), so `loss.backward()` of user-written losses runs on the library too.  Under
`create_graph=True` that backward is itself differentiable once more (`dmip_mlp_double_backward`: derivative terms such as
the reference's Score-FPE divergence and ds/dt, losses.py:14-40, train the net), for cotangents on the input gradient and
on the incoming gradient; a cotangent on a parameter gradient (NotImplementedError) and a third derivative
(RuntimeError) raise.  Nets outside the shapes those
kernels serve fall back to the torch module chain (twice differentiable) with a RuntimeWarning.
`GaussianFourierProjection` / `TemporalMLP*` of the reference are unused by every model (nets.py:62-63) and omitted.
"""
import ctypes as C
import warnings

import torch
from torch import nn

from . import _lib

_WARNED_EAGER = [False]


class DmipMlpGrad(C.Structure):
    _fields_ = [("net", _lib.DmipMlp), ("n", C.c_int64), ("x_dim", C.c_int32), ("cond_dim", C.c_int32),
                ("x", C.c_void_p), ("cond", C.c_void_p), ("t", C.c_void_p), ("out", C.c_void_p),
                ("grad_out", C.c_void_p), ("grad_params", C.c_void_p), ("grad_in", C.c_void_p),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t)]


class DmipMlpGradGrad(C.Structure):
    _fields_ = [("net", _lib.DmipMlp), ("n", C.c_int64), ("x_dim", C.c_int32), ("cond_dim", C.c_int32),
                ("x", C.c_void_p), ("cond", C.c_void_p), ("t", C.c_void_p), ("grad_out", C.c_void_p),
                ("gg_in", C.c_void_p), ("gg_out", C.c_void_p), ("grad_params", C.c_void_p), ("grad_in", C.c_void_p),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t)]


def _bind_grad():
    L = _lib.require_gpu()
    if not getattr(L, "_mlp_grad_bound", False):
        L.dmip_mlp_grad_workspace_bytes.restype = C.c_size_t
        L.dmip_mlp_grad_workspace_bytes.argtypes = [C.POINTER(DmipMlpGrad)]
        L.dmip_mlp_forward_stash.restype = C.c_int
        L.dmip_mlp_forward_stash.argtypes = [C.POINTER(DmipMlpGrad), C.c_void_p]
        L.dmip_mlp_backward.restype = C.c_int
        L.dmip_mlp_backward.argtypes = [C.POINTER(DmipMlpGrad), C.c_void_p]
        L.dmip_loss_grad_floats.restype = C.c_size_t
        L.dmip_loss_grad_floats.argtypes = [C.POINTER(_lib.DmipMlp)]
        L.dmip_mlp_double_backward_workspace_bytes.restype = C.c_size_t
        L.dmip_mlp_double_backward_workspace_bytes.argtypes = [C.POINTER(DmipMlpGradGrad)]
        L.dmip_mlp_double_backward.restype = C.c_int
        L.dmip_mlp_double_backward.argtypes = [C.POINTER(DmipMlpGradGrad), C.c_void_p]
        L._mlp_grad_bound = True
    return L


def _grad_desc(net, x, cond, t, keep):
    d = DmipMlpGrad()
    d.net = _lib.mlp_desc(net, keep)
    d.n = x.shape[0]
    d.x_dim = x.shape[1]
    d.x, d.t = x.data_ptr(), t.data_ptr()
    if cond is not None:
        d.cond_dim = cond.shape[1]
        d.cond = cond.data_ptr()
    return d


def _mlp_backward(ctx, gout):
    """`dmip_mlp_backward` over the stash of `_MlpFn.forward`: (gradient w.r.t. cat[x, cond, t] or None, flat parameter
    gradient [W_0, b_0, W_1, b_1, ...])."""
    L = _bind_grad()
    d = ctx.d
    dev = gout.device
    flat = torch.empty(L.dmip_loss_grad_floats(C.byref(d.net)), device=dev, dtype=torch.float32)
    need_in = any(ctx.needs_input_grad[1:4])
    gin = torch.empty(gout.shape[0], d.net.in_dim, device=dev, dtype=torch.float32) if need_in else None
    d.grad_out, d.grad_params = gout.data_ptr(), flat.data_ptr()
    d.grad_in = gin.data_ptr() if need_in else None
    with torch.cuda.device(dev):
        _lib.check(L.dmip_mlp_backward(C.byref(d), _lib.stream_ptr()))
    return gin, flat


class _MlpFn(torch.autograd.Function):
    """a(x, cond, t) with a backward on the library's own kernels (`dmip_mlp_forward_stash` / `dmip_mlp_backward`,
    include/dmip.h): what `loss.backward()` of a user-written loss runs instead of torch's addmm / tanh chain.
    Under `create_graph=True` the backward runs as `_MlpGradFn`, whose own backward is `dmip_mlp_double_backward`."""

    @staticmethod
    def forward(ctx, net, x, cond, t, *params):
        L = _bind_grad()
        keep = [x, cond, t]
        d = _grad_desc(net, x, cond, t, keep)
        out = torch.empty(x.shape[0], net.output_dim, device=x.device, dtype=torch.float32)
        d.out = out.data_ptr()
        nbytes = L.dmip_mlp_grad_workspace_bytes(C.byref(d))
        ws = torch.empty(nbytes + 1024, dtype=torch.uint8, device=x.device)
        d.workspace = (ws.data_ptr() + 1023) & ~1023
        d.workspace_bytes = nbytes
        with torch.cuda.device(x.device):
            _lib.check(L.dmip_mlp_forward_stash(C.byref(d), _lib.stream_ptr()))
        ctx.d, ctx.keep, ctx.ws = d, keep, ws
        ctx.net = net
        ctx.shapes = [p.shape for p in params]
        ctx.dims = (x.shape[1], 0 if cond is None else cond.shape[1])
        ctx.save_for_backward(x, cond, t, *params)        # read only by a create_graph=True backward
        net.last_launch_count = L.dmip_last_launch_count()
        return out

    @staticmethod
    def backward(ctx, gout):
        gout = gout.contiguous().float()
        if torch.is_grad_enabled():
            # create_graph=True: the same backward, recorded as a differentiable op
            x, cond, t, *params = ctx.saved_tensors
            gin, flat = _MlpGradFn.apply(ctx, gout, x, cond, t, *params)
        else:
            gin, flat = _mlp_backward(ctx, gout)
        grads, off = [], 0
        for shp in ctx.shapes:
            grads.append(flat[off:off + shp.numel()].view(shp))
            off += shp.numel()
        need_in = gin is not None
        xd, cd = ctx.dims
        gx = gin[:, :xd] if need_in and ctx.needs_input_grad[1] else None
        gc = gin[:, xd:xd + cd] if need_in and cd and ctx.needs_input_grad[2] else None
        gt = gin[:, xd + cd:].reshape(ctx.keep[2].shape) if need_in and ctx.needs_input_grad[3] else None
        return (None, gx, gc, gt, *grads)


class _MlpGradFn(torch.autograd.Function):
    """The backward of `_MlpFn` as a function of (u = grad_out, x, cond, t, params) -> (input gradient, flat parameter
    gradient), differentiated by `dmip_mlp_double_backward` (include/dmip.h): a cotangent v on the input gradient gives
    J v for u, and for the inputs and parameters the gradient of u^T J v.  Parameter-space cotangents (Hessian-vector
    products in parameter space) and third order are not provided: both raise."""

    @staticmethod
    def forward(ctx, fctx, gout, x, cond, t, *params):
        ctx.set_materialize_grads(False)
        ctx.fctx = fctx
        ctx.save_for_backward(gout, x, cond, t, *params)
        return _mlp_backward(fctx, gout)

    @staticmethod
    def backward(ctx, g_gin, g_flat):
        if g_flat is not None:
            raise NotImplementedError(
                "dmip score nets: the parameter gradient of MLP.forward is not differentiable (no Hessian-vector products "
                "in parameter space); only the input gradient and the incoming gradient carry a second derivative")
        with torch.no_grad():
            res = _mlp_double_backward(ctx, g_gin)
        if torch.is_grad_enabled():
            # create_graph=True: these results depend on u, x, cond, t, the parameters and v, but no kernel differentiates
            # them again — route them through a node that refuses, connected to every one of those that requires grad,
            # instead of letting them pass as constants (a silently wrong third derivative)
            live = [i for i, r in enumerate(res) if r is not None]
            anchors = [a for a in list(ctx.saved_tensors) + [g_gin] if a is not None and a.requires_grad]
            if live and anchors:
                out = _ThirdOrderRefused.apply(len(live), *[res[i] for i in live], *anchors)
                out = out if isinstance(out, tuple) else (out,)
                res = list(res)
                for i, r in zip(live, out):
                    res[i] = r
                res = tuple(res)
        return res


def _mlp_double_backward(ctx, g_gin):
    """`dmip_mlp_double_backward` for `_MlpGradFn.backward`: the gradients of <v, J^T u> = u^T J v, v = g_gin, w.r.t. the
    inputs of `_MlpGradFn` (None where not needed)."""
    n_params = len(ctx.fctx.shapes)
    if g_gin is None:
        return (None,) * (5 + n_params)
    L = _bind_grad()
    gout, x, cond, t = ctx.saved_tensors[:4]
    fctx = ctx.fctx
    need_u = ctx.needs_input_grad[1]
    need_in = any(ctx.needs_input_grad[2:5])
    need_p = any(ctx.needs_input_grad[5:])
    dev = gout.device
    n = gout.shape[0]
    v = g_gin.contiguous().float()
    d = DmipMlpGradGrad()
    d.net = fctx.d.net                                  # the weights of the forward (kept alive by fctx.keep)
    d.n, d.x_dim, d.cond_dim = fctx.d.n, fctx.d.x_dim, fctx.d.cond_dim
    d.x, d.cond, d.t = fctx.d.x, fctx.d.cond, fctx.d.t
    d.grad_out, d.gg_in = gout.data_ptr(), v.data_ptr()
    guard = _lib.Guarded()                              # DMIP_GUARD=1: canaries around every buffer the kernels write
    gg_out = guard.empty(n * d.net.out_dim, torch.float32, dev).view(n, d.net.out_dim) if need_u else None
    gin = guard.empty(n * d.net.in_dim, torch.float32, dev).view(n, d.net.in_dim) if need_in else None
    flat = guard.empty(L.dmip_loss_grad_floats(C.byref(d.net)), torch.float32, dev) if need_p else None
    for name, buf in (("gg_out", gg_out), ("grad_in", gin), ("grad_params", flat)):
        setattr(d, name, None if buf is None else buf.data_ptr())
    nbytes = L.dmip_mlp_double_backward_workspace_bytes(C.byref(d))
    ws = guard.empty(nbytes + 1024, torch.uint8, dev)
    d.workspace = (ws.data_ptr() + 1023) & ~1023
    d.workspace_bytes = nbytes
    with torch.cuda.device(dev):
        _lib.check(L.dmip_mlp_double_backward(C.byref(d), _lib.stream_ptr()))
    guard.check("dmip_mlp_double_backward")
    fctx.net.last_launch_count = L.dmip_last_launch_count()
    grads = [None] * n_params
    if need_p:
        off = 0
        for i, shp in enumerate(fctx.shapes):
            grads[i] = flat[off:off + shp.numel()].view(shp)
            off += shp.numel()
    xd, cd = fctx.dims
    gx = gin[:, :xd] if need_in and ctx.needs_input_grad[2] else None
    gc = gin[:, xd:xd + cd] if need_in and cd and ctx.needs_input_grad[3] else None
    gt = gin[:, xd + cd:].reshape(t.shape) if need_in and ctx.needs_input_grad[4] else None
    return (None, gg_out, gx, gc, gt, *grads)


THIRD_ORDER_MSG = ("dmip score nets: MLP.forward is differentiable twice, not three times (dmip_mlp_double_backward has no "
                   "backward of its own)")


class _ThirdOrderRefused(torch.autograd.Function):
    """Identity on the first `n` tensors (the results of `dmip_mlp_double_backward` under create_graph=True), recorded as a
    function of the tensors they depend on (`anchors`); differentiating them raises."""

    @staticmethod
    def forward(ctx, n, *tensors):
        return tensors[:n] if n > 1 else tensors[0]

    @staticmethod
    def backward(ctx, *cotangents):
        raise RuntimeError(THIRD_ORDER_MSG)


class _ScoreMLP(nn.Sequential):
    """[in] -> hidden... -> [out] tanh MLP with the reference's module naming."""

    def __init__(self, input_dim, output_dim, hidden_layers, activation):
        super().__init__()
        self.input_dim = input_dim
        self.output_dim = output_dim
        self.hidden_layers = hidden_layers
        widths = [input_dim] + list(hidden_layers)
        self.add_module('0', nn.Linear(widths[0], widths[1]))
        self.add_module('1', activation)
        self.add_module('act', activation)          # second registration of the same module: double tanh (Q1)
        for fan_in, fan_out in zip(widths[1:-1], widths[2:]):
            self.add_module(str(len(self)), nn.Linear(fan_in, fan_out))
            self.add_module(str(len(self)), activation)
        self.add_module(str(len(self)), nn.Linear(widths[-1], output_dim))
        self._packed = _lib.PackedNet()
        self.precision = 'bf16'
        self.l0_split = 4                    # layer-0 operand: one f16 part (1: bf16, 2: bf16 hi + lo, 3: + W0 split)

    def _fused(self, x, cond, t):
        L = _lib.require_gpu()
        n = x.shape[0]
        keep = []
        d = _lib.DmipForward()
        d.net = _lib.mlp_desc(self, keep)
        prec = _lib.precision_code(self.precision)
        if prec == _lib.PREC_BF16 and not _lib.tc_supported(self, None, self.l0_split):
            prec = _lib.PREC_F32                     # other widths / too deep a layer 0: fp32 FFMA kernels (still CUDA, never CPU)
        self.last_precision = 'bf16' if prec == _lib.PREC_BF16 else 'fp32'   # the path that actually ran
        d.precision = prec
        d.l0_split = self.l0_split
        d.n = n
        x = x.detach().float().contiguous()
        t = t.detach().float().reshape(-1).contiguous()
        assert t.numel() == n, 'Input Tensor is expected to be 2D with shape (batch_size, xdim+ydim+1)'
        d.x_dim = x.shape[1]
        d.x = x.data_ptr()
        d.t = t.data_ptr()
        if cond is not None and cond.numel() > 0:
            cond = cond.detach().float().contiguous()
            d.cond_dim = cond.shape[1]
            d.cond = cond.data_ptr()
        out = torch.empty(n, self.output_dim, device=x.device, dtype=torch.float32)
        d.out = out.data_ptr()
        with torch.cuda.device(x.device):            # launch on the tensors' device and its current stream
            if prec == _lib.PREC_BF16:
                d.packed = self._packed.get(self, d.net.in_dim, self.output_dim, self.l0_split).data_ptr()
            else:
                ws = torch.empty(max(L.dmip_forward_workspace_bytes(C.byref(d)), 16), dtype=torch.uint8, device=x.device)
                keep.append(ws)
                d.workspace = ws.data_ptr()
                d.workspace_bytes = ws.numel()
            _lib.check(L.dmip_mlp_forward(C.byref(d), _lib.stream_ptr()))
        return out

    def _autograd_fused(self, x, cond, t):
        """Autograd through the library's own kernels (forward with stash + backward), or None when the net's shape is
        outside what they serve."""
        L = _bind_grad()
        if x.shape[0] == 0:
            return None
        xx = x.float().contiguous()
        cc = None if cond is None or cond.numel() == 0 else cond.float().contiguous()
        tt = t.float().reshape(-1).contiguous()
        assert tt.numel() == xx.shape[0], 'Input Tensor is expected to be 2D with shape (batch_size, xdim+ydim+1)'
        probe = _grad_desc(self, xx.detach(), None if cc is None else cc.detach(), tt.detach(), [])
        if L.dmip_mlp_grad_workspace_bytes(C.byref(probe)) == 0:
            return None
        params = [p for lin in _lib.linear_layers(self) for p in (lin.weight, lin.bias)]
        return _MlpFn.apply(self, xx, cc, tt, *params)

    def invalidate_packed(self):
        """Drop the cached tcgen05 weight image (needed only after writes through `p.data`, see _lib.PackedNet)."""
        self._packed.invalidate()

    def _dispatch(self, x, cond, t):
        params_need_grad = torch.is_grad_enabled() and (
            x.requires_grad or t.requires_grad or (cond is not None and cond.requires_grad)
            or any(p.requires_grad for p in self.parameters()))
        if x.is_cuda and not params_need_grad:
            return self._fused(x, cond, t)
        if not x.is_cuda:
            raise RuntimeError("dmip score nets run on CUDA (sm_100a) only: there is no CPU fallback")
        fused = self._autograd_fused(x, cond, t)
        if fused is not None:
            return fused
        if not _WARNED_EAGER[0]:
            _WARNED_EAGER[0] = True
            warnings.warn("dmip: autograd is recording through MLP.forward of a net the tcgen05 kernels do not serve (they take "
                          "[in <= 64] -> 512 -> 512 -> 512 -> [out <= 64]) — this call runs the plain torch module chain "
                          "(cuBLAS addmm), not the fused sm_100a kernels.", RuntimeWarning, stacklevel=3)
        parts = [x] + ([cond] if cond is not None and cond.numel() > 0 else []) + [t.view(len(x), 1)]
        inp = torch.cat(parts, dim=1)
        assert inp.ndim == 2, 'Input Tensor is expected to be 2D with shape (batch_size, xdim+ydim+1)'
        return nn.Sequential.forward(self, inp)


class MLP(_ScoreMLP):
    """a(x, y, t) on cat[x, y, t]; `y` may be the empty tensor (CDiffE losses)."""

    def forward(self, x, y, t):
        return self._dispatch(x, y, t)


class MLP2(_ScoreMLP):
    """s(x, t) on cat[x, t] — the DPS prior net."""

    def forward(self, x, t):
        return self._dispatch(x, None, t)


class PosteriorScore(nn.Module):
    """g(t, x) * (prior_net(x, t) + likelihood_net(x, y, t)) — the DPS drift."""

    def __init__(self, prior_net, likelihood_net, forward_process):
        super().__init__()
        self.prior_net = prior_net
        self.likelihood_net = likelihood_net
        self.forward_sde = forward_process

    def forward(self, x, y, t):
        return self.forward_sde.g(t, x) * (self.prior_net(x, t) + self.likelihood_net(x, y, t))
