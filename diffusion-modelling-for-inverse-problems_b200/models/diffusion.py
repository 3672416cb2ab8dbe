"""Drop-in for the reference's `models/diffusion.py`: CDE, CDiffE (Batzolis et al. 2021) and
PosteriorDiffusionEstimator (after Chung et al. 2022), same constructors, attributes and call signatures:

    model = CDE(xdim, ydim, hidden_layers)
    x = model(y, num_samples=2000, num_steps=200, mean=0, std=1)      # np.ndarray (num_samples, xdim) float32
    loss, info = model.train_epoch(optimizer, loss_fn, epoch_data_loader)
    model.sde, model.sde.a, model.sde.base_sde, model.sde.T, model.sde.debias

`forward` replaces the reference's S x ~30-kernel Python loop (models/diffusion.py:38-42, :171-177) by ONE launch of
the persistent fused Euler–Maruyama kernel (`dmip_sampler_em_vp`, include/dmip.h).  Extras beyond the reference
signature are keyword-only: `precision` ('bf16' tcgen05 path | 'fp32' FFMA path), `seed` (Philox key; the
reference uses torch's global RNG, which a fused kernel cannot consume — statistics are preserved, streams differ),
`injected` (dict with 'x0', 'noise'[, 'ynoise'] standard-normal tensors: bit-for-bit the reference's draws, for
parity tests), `gidx_base` (global particle offset for multi-GPU sharding), `return_tensor`, `n_corrector` / `snr`
(Langevin corrector sub-steps after every predictor step: the predictor–corrector sampler of Song et al. 2021; 0 = the
reference's Euler–Maruyama predictor).  A model built with `base_sde=sdes.VarianceExplodingSDE(...)` samples the VE-SDE.  `y` may also be a
batch (n_obs, ydim): all observations are integrated in the same launch and (n_obs, num_samples, xdim) is returned.

CDiffE.forward upstream raises TypeError (it omits `cond` when calling `sde.mu`, SURVEY.md Q7); the intended call
(`cond` = empty tensor, as the loss path does) is what is implemented here.
"""
import ctypes as C
import weakref

import torch
from torch import nn

from .. import _lib
from .. import sdes
from ..distributed import GraphedTrainStep, _bucket_nets, fused_optimizer_step
from ..losses import PosteriorLoss, fused_train_step
from ..nets import MLP, MLP2, PosteriorScore

device = 'cuda' if torch.cuda.is_available() else 'cpu'

_VARIANT = {'CDE': _lib.CDE, 'CDiffE': _lib.CDIFFE, 'Posterior': _lib.DPS}


def _owns_all_grads(model, optimizer):
    """True when `optimizer.zero_grad(); loss.backward(); optimizer.step()` can be replaced by the fused step that writes
    the gradient straight into the parameters' `.grad` (dmip.distributed.fused_optimizer_step): every parameter of the
    optimizer is a trainable parameter of the model's score net(s) without gradient hooks — nothing else would get, or
    keep, a gradient from this loss.  The verdict is cached ON the optimizer (for this model and parameter count)."""
    key = (id(model), sum(len(g['params']) for g in optimizer.param_groups))
    hit = optimizer.__dict__.get('_dmip_fused_step_ok')
    if hit is None or hit[0] != key:
        mine = {id(p): p for net in _bucket_nets(model) for lin in _lib.linear_layers(net) for p in (lin.weight, lin.bias)}
        theirs = [p for g in optimizer.param_groups for p in g['params']]
        ok = (len(theirs) == len(mine) and all(id(p) in mine for p in theirs)
              and all(p.requires_grad and not p._backward_hooks and p.is_cuda for p in mine.values()))
        hit = optimizer.__dict__['_dmip_fused_step_ok'] = (key, ok)
    return hit[1]


class BaseClassDiffusionModel():

    variant = 'CDE'

    def __init__(self, xdim, ydim):
        self.xdim = xdim
        self.ydim = ydim
        self.sde = None                      # set by subclasses
        self.precision = 'bf16'
        self.l0_split = 4                    # layer-0 operand: one f16 part (1: bf16, 2: bf16 hi + lo, 3: + W0 split)
        self._packed = (_lib.PackedNet(), _lib.PackedNet())
        self._seed_counter = 0
        self._stage = None                   # pinned host staging buffer of the sampler's result

    def __call__(self, *args, **kwargs):
        return self.forward(*args, **kwargs)

    # ------------------------------------------------------------------ sampling
    def _nets(self):
        """(net, net2): score net; for DPS (likelihood_net, prior_net)."""
        return self.sde.a, None

    def forward(self, y, num_samples=2000, num_steps=200, mean=0, std=1, *, precision=None, seed=None,
                injected=None, gidx_base=0, return_tensor=False, n_corrector=0, snr=0.16):
        L = _lib.require_gpu()
        net, net2 = self._nets()
        dev = next(net.parameters()).device
        if dev.type != 'cuda':
            raise RuntimeError("dmip samplers run on CUDA (sm_100a) only: move the model to the GPU (no CPU fallback)")
        y = torch.as_tensor(y, dtype=torch.float32)
        batched = y.ndim == 2
        ys = y.reshape(-1, self.ydim).to(dev).contiguous()
        n_obs = ys.shape[0]
        n_total = n_obs * num_samples

        keep = [ys]
        d = _lib.DmipSampler()
        d.variant = _VARIANT[self.variant]
        prec = _lib.precision_code(self.precision if precision is None else precision)
        dv = self.xdim + self.ydim if self.variant == 'CDiffE' else self.xdim
        if prec == _lib.PREC_BF16 and not (_lib.tc_supported(net, dv, self.l0_split)
                                            and (net2 is None or _lib.tc_supported(net2, self.xdim, self.l0_split))
                                            and (net2 is None or self.xdim <= 8) and self.xdim <= 104
                                            and (self.variant != 'CDiffE' or (self.xdim <= 32 and self.ydim <= 24))):
            prec = _lib.PREC_F32             # other layer widths / state sizes: fp32 FFMA kernels (still CUDA, never CPU)
        d.precision = prec
        self.last_precision = 'bf16' if prec == _lib.PREC_BF16 else 'fp32'   # the path that actually ran (bench.py's dtype)
        d.xdim, d.ydim = self.xdim, self.ydim
        d.n_obs, d.n_per_obs, d.num_steps = n_obs, num_samples, num_steps
        d.T = float(self.sde.T)
        _lib.set_sde(d, self.sde.base_sde)                                 # VP, or VE beyond the reference
        d.n_corrector, d.snr = int(n_corrector), float(snr)
        n_sub = num_steps * (1 + int(n_corrector))                         # sub-steps: predictor + Langevin correctors
        d.mean, d.std = float(mean), float(std)
        d.net = _lib.mlp_desc(net, keep)
        if net2 is not None:
            d.net2 = _lib.mlp_desc(net2, keep)
        d.l0_split = self.l0_split
        d.y = ys.data_ptr()
        guard = _lib.Guarded()
        out = guard.empty(n_total * self.xdim, torch.float32, dev).view(n_total, self.xdim)
        d.out = out.data_ptr()
        if injected is not None:
            d.rng_mode = _lib.RNG_INJECTED
            for name in ('x0', 'noise') + (('ynoise',) if self.variant == 'CDiffE' else ()):
                tns = injected[name].to(dev, torch.float32).contiguous()
                keep.append(tns)
                setattr(d, name, tns.data_ptr())
            assert injected['x0'].numel() == n_total * self.xdim, 'x0 must have shape (n_obs*num_samples, xdim)'
            assert injected['noise'].numel() == n_sub * n_total * self.xdim, 'noise must be (S * (1 + n_corrector), N, xdim)'
        else:
            d.rng_mode = _lib.RNG_PHILOX
            if seed is None:                 # fresh stream per call, like successive draws from a global RNG
                seed = (torch.initial_seed() + 0x9E3779B97F4A7C15 * (self._seed_counter + 1)) & (2 ** 64 - 1)
                self._seed_counter += 1
            d.seed = int(seed) & (2 ** 64 - 1)
        d.gidx_base = int(gidx_base)
        with torch.cuda.device(dev):
            if prec == _lib.PREC_BF16:
                d.packed = self._packed[0].get(net, dv, self.xdim, self.l0_split).data_ptr()
                if net2 is not None:
                    d.packed2 = self._packed[1].get(net2, self.xdim, self.xdim, self.l0_split).data_ptr()
            ws = torch.empty(max(L.dmip_sampler_workspace_bytes(C.byref(d)), 16), dtype=torch.uint8, device=dev)
            keep.append(ws)
            d.workspace = ws.data_ptr()
            d.workspace_bytes = ws.numel()
            _lib.check(L.dmip_sampler_em_vp(C.byref(d), _lib.stream_ptr()))
            self.last_launch_count = L.dmip_last_launch_count()
            guard.check("dmip_sampler_em_vp")
        if batched:
            out = out.view(n_obs, num_samples, self.xdim)
        if return_tensor:
            return out
        return self._to_host(out, dev)

    _PINNED_POOL_BYTES = 4 << 30

    def _to_host(self, out, dev):
        """The reference's single device->host crossing (models/diffusion.py:44).  The samples are DMA-ed straight into a
        pinned buffer that IS the returned array's memory (no host-side copy): buffers are pooled and one is reused as
        soon as the array handed out earlier has been dropped (a weak reference to that array tells).
        A caller that keeps every result alive gets fresh pinned buffers up to _PINNED_POOL_BYTES, then pageable memory
        filled through two 32 MB pinned staging chunks.  (A pageable .cpu() of 1M x 100 samples costs 0.2 s, this 0.01 s.)"""
        n = out.numel()
        stream = torch.cuda.current_stream(dev)
        if self._stage is None:
            self._stage = {'pool': [], 'chunks': None}
        pool = self._stage['pool']
        ent = next((e for e in pool if e[0].numel() >= n and (e[1] is None or e[1]() is None)), None)
        if ent is None and 4 * (sum(e[0].numel() for e in pool) + n) <= self._PINNED_POOL_BYTES:
            ent = [torch.empty(max(n, 1), dtype=torch.float32, pin_memory=True), None]
            pool.append(ent)
        if ent is not None:
            view = ent[0][:n].view(out.shape)
            view.copy_(out, non_blocking=True)
            stream.synchronize()
            arr = view.numpy()
            ent[1] = weakref.ref(arr)                # views derived from it keep it alive through .base
            return arr
        flat = out.reshape(-1)
        chunk = 8 << 20
        if self._stage['chunks'] is None:
            self._stage['chunks'] = ([torch.empty(chunk, dtype=torch.float32, pin_memory=True) for _ in range(2)],
                                     [torch.cuda.Event() for _ in range(2)])
        bufs, evs = self._stage['chunks']
        host = torch.empty(n, dtype=torch.float32)
        n_chunks = (n + chunk - 1) // chunk
        for c in range(n_chunks + 1):
            if c < n_chunks:
                lo, hi = c * chunk, min(n, (c + 1) * chunk)
                bufs[c & 1][:hi - lo].copy_(flat[lo:hi], non_blocking=True)
                evs[c & 1].record(stream)
            if c >= 1:
                lo, hi = (c - 1) * chunk, min(n, c * chunk)
                evs[(c - 1) & 1].synchronize()
                host[lo:hi].copy_(bufs[(c - 1) & 1][:hi - lo])
        return host.view(out.shape).numpy()

    def invalidate_packed(self):
        """Drop the cached tcgen05 weight images (needed only after writes through `p.data`, see _lib.PackedNet)."""
        for p in self._packed:
            p.invalidate()

    # ------------------------------------------------------------------ training
    def sample_t(self, x, eps=1e-4):
        base = self.sde.base_sde
        if x.is_cuda and hasattr(base, 'sample_t_device'):
            # the reference draws t on the CPU and copies it over every batch; at its own batch size that is a third of
            # the step's host time — same distribution, drawn where it is used
            t_ = base.sample_t_device([x.size(0), ] + [1 for _ in range(x.ndim - 1)], x.device, self.sde.debias, eps)
            t_ = t_.to(x.dtype)
            t_.requires_grad = True
            return t_
        if self.sde.debias:
            t_ = self.sde.base_sde.sample_debiasing_t([x.size(0), ] + [1 for _ in range(x.ndim - 1)]) + eps
            t_ = torch.where(t_ > self.sde.T, t_ - eps, t_).to(x)
        else:
            t_ = eps + torch.rand([x.size(0), ] + [1 for _ in range(x.ndim - 1)]).to(x) * self.sde.T
            t_ = torch.where(t_ > self.sde.T, torch.full_like(t_, self.sde.T - eps), t_)
        t_.requires_grad = True
        return t_

    def _graphed_step_for(self, optimizer, loss_fn, x, y):
        """The captured step for this (optimizer, loss, batch shape): captured on first sight; a batch of another shape
        (the ragged last one of an epoch) runs eagerly unless that shape comes back, which replaces the capture."""
        if len(optimizer.state) == 0:
            return None       # the optimizer creates its state on its first step: that step runs eagerly, outside any capture
        key = GraphedTrainStep.key_of(optimizer, loss_fn, x, y)
        gs = self.__dict__.get('_graphed_step')
        if gs is not None and gs.key == key:
            return gs
        if gs is None or self.__dict__.get('_graph_miss') == key:
            self._graphed_step = GraphedTrainStep(self, optimizer, loss_fn, x, y)
            return self._graphed_step
        self._graph_miss = key
        return None

    def train_epoch(self, optimizer, loss_fn, epoch_data_loader, *, graph=False):
        """Upstream's epoch loop.  graph=True (keyword-only extra): batches of a repeating shape run as one CUDA-graph
        replay each (dmip.distributed.GraphedTrainStep — the launch-bound regime of small batches); anything the graph
        cannot serve (other shapes, an optimizer with foreign parameters) takes the eager path below."""
        mean_loss = 0
        logger_info = {}
        for k, (x, y) in enumerate(epoch_data_loader()):
            fused_ok = x.is_cuda and _owns_all_grads(self, optimizer)
            replay = self._graphed_step_for(optimizer, loss_fn, x, y) if graph and fused_ok else None
            if replay is not None:
                loss, loss_info = replay(x, y)
                stepped = True
            elif fused_ok:
                # zero_grad / backward / step without the autograd round trip (dmip.distributed.fused_optimizer_step)
                loss, loss_info = fused_optimizer_step(self, optimizer, loss_fn, x, y, self.sample_t(x))
                stepped = True
            else:
                loss, loss_info = fused_train_step(self, loss_fn, x, y, self.sample_t(x))
                stepped = False
            # running means as upstream (models/diffusion.py:90-92, :103), kept on the device in float64 — the arithmetic
            # of upstream's Python floats — as ONE vector, and read back once per epoch instead of one .item() per
            # entry per batch
            if loss_info:
                keys = list(loss_info)
                vals = torch.stack([loss_info[key].detach() for key in keys]).double()
                logger_info = (logger_info * k / (k + 1) if k else 0) + vals / (k + 1)
            if not stepped:
                optimizer.zero_grad()
                loss.backward()
                optimizer.step()
            mean_loss = mean_loss * k / (k + 1) + loss.detach() / (k + 1)
        if not torch.is_tensor(logger_info):
            return mean_loss, {}
        return mean_loss, dict(zip(keys, logger_info.tolist()))


class CDE(BaseClassDiffusionModel):
    """Conditional denoising estimator: score net a(x_t, y, t) -> xdim."""

    variant = 'CDE'

    def __init__(self, xdim, ydim, hidden_layers, *, base_sde=None):
        super().__init__(xdim, ydim)
        score_net = MLP(input_dim=xdim + ydim + 1, output_dim=xdim, hidden_layers=hidden_layers,
                        activation=nn.Tanh()).to(device)
        self.sde = sdes.PluginReverseSDE(base_sde or sdes.VariancePreservingSDE(), score_net, T=1, debias=True)


class CDiffE(BaseClassDiffusionModel):
    """Conditional diffusive estimator: joint score of z = [x, y]; y is re-diffused at every sampling step."""

    variant = 'CDiffE'

    def __init__(self, xdim, ydim, hidden_layers, *, base_sde=None):
        super().__init__(xdim, ydim)
        score_net = MLP(input_dim=xdim + ydim + 1, output_dim=xdim + ydim, hidden_layers=hidden_layers,
                        activation=nn.Tanh()).to(device)
        self.sde = sdes.PluginReverseSDE(base_sde or sdes.VariancePreservingSDE(), score_net, T=1, debias=True)


class PosteriorDiffusionEstimator(BaseClassDiffusionModel):
    """Diffusion posterior sampler: drift = g * (prior_net(x,t) + likelihood_net(x,y,t))."""

    variant = 'Posterior'

    def __init__(self, xdim, ydim, hidden_layers, *, base_sde=None):
        super().__init__(xdim, ydim)
        forward_process = base_sde or sdes.VariancePreservingSDE()
        prior_net = MLP2(input_dim=xdim + 1, output_dim=xdim, hidden_layers=hidden_layers,
                         activation=nn.Tanh()).to(device)
        likelihood_net = MLP(input_dim=xdim + ydim + 1, output_dim=xdim, hidden_layers=hidden_layers,
                             activation=nn.Tanh()).to(device)
        score_net = PosteriorScore(prior_net, likelihood_net, forward_process)
        self.sde = sdes.PluginReverseSDE(forward_process, score_net, T=1, debias=True)
        self.loss_fn = PosteriorLoss

    def _nets(self):
        return self.sde.a.likelihood_net, self.sde.a.prior_net
