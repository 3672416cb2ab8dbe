"""The numbers of the reference's `evaluate` loops (main_diffusion_linear.py:53-137,
main_diffusion_scatterometry.py:40-124) computed where the samples are: histogram KL (both directions), negative
log-likelihood of model and ground-truth samples, and the MSE of the learned score at t = 0.

Upstream loops over the test observations one by one — a 5 000-particle sampler call each, `np.histogramdd` on the
host, a D2H copy per call.  Here all observations of a repeat are ONE sampler launch (`model(ys, ...)` with a batch of
observations, 5 000 x n_obs particles), the samples stay on the GPU (`return_tensor=True`), histograms/KL run in
`dmip.metrics`, the score net in the fused forward.  Plots are not produced (no matplotlib in this image); the
per-observation table the reference writes to results.csv is returned and optionally written.

Beyond the reference, `mmd_bandwidths=(...)` adds a per-observation 'MMD' column: the unbiased MMD^2 between the
ground-truth and the model samples for the sum of the Gaussian kernels of those bandwidths, averaged over repeats (one
batched `metrics.mmd2` call per repeat).  `ksd_scales=(...)` adds two columns: the IMQ kernel Stein discrepancy
KSD^2_U of the ground-truth samples ('KSD_true' for the exact linear posterior — the estimator's noise floor —,
'KSD_mcmc' for the Metropolis chains) and of the model samples ('KSD_diffusion') against the exact posterior score,
summed over those scales and averaged over repeats.  It needs no ground truth, so it grades the Metropolis reference
samples on the same scale as the model.  Without these keywords the tables are the reference's.
"""
import os

import numpy as np
import torch

from . import metrics
from .utils_scatterometry import get_log_posterior


def _finish(table, out_dir):
    if out_dir is not None:
        import pandas as pd
        os.makedirs(out_dir, exist_ok=True)
        pd.DataFrame(table).to_csv(os.path.join(out_dir, 'results.csv'))
    return table


def _score_mse(model, x_true, ys):
    """mean_n sum_d (a(x, y, 0)/g(0) - score_true)^2 needs a(x, y, 0)/g(0) for (n_obs, n, xdim) ground-truth samples"""
    n_obs, n, xdim = x_true.shape
    flat = x_true.reshape(-1, xdim)
    yy = ys[:, None, :].expand(n_obs, n, ys.shape[1]).reshape(n_obs * n, -1)
    t0 = torch.zeros(n_obs * n, 1, device=flat.device)
    g0 = model.sde.base_sde.g(t0, flat)
    with torch.no_grad():
        return model.sde.a(flat, yy, t0) / g0, flat, yy


class _RunningMean:
    """Running mean over repeats of a per-observation metric (a CUDA tensor (n_obs,) per repeat)."""

    def __init__(self):
        self.total = None
        self.n = 0

    def add(self, v):
        self.total = v if self.total is None else self.total + v
        self.n += 1

    def mean(self):
        return (self.total / self.n).cpu().numpy()


class _MixtureMMD(_RunningMean):
    """Running mean over repeats of MMD^2_u for the summed kernel sum_b k_b (MMD^2 is linear in the kernel)."""

    def __init__(self, bandwidths):
        super().__init__()
        self.bandwidths = tuple(float(b) for b in bandwidths)

    def add(self, x_true, x_pred):
        super().add(metrics.mmd2(x_true, x_pred, self.bandwidths).sum(-1))


class _SteinKSD:
    """Running means over repeats of the IMQ KSD^2_U, summed over `scales`, of the ground-truth and the model samples
    (n_obs, n, d) against the exact posterior score score_fn(x, y) of flattened rows."""

    def __init__(self, scales, score_fn):
        self.scales = tuple(float(c) for c in scales)
        self.score_fn = score_fn
        self.true, self.model = _RunningMean(), _RunningMean()

    def _ksd(self, x, score):
        return metrics.ksd2(x, score.reshape(x.shape), self.scales).sum(-1)

    def add(self, x_true, score_true, x_pred, ys):
        """score_true: the score at the rows of x_true, already computed by the caller"""
        n_obs, n, d = x_pred.shape
        yy = ys[:, None, :].expand(n_obs, n, ys.shape[1]).reshape(n_obs * n, -1)
        self.true.add(self._ksd(x_true, score_true))
        self.model.add(self._ksd(x_pred, self.score_fn(x_pred.reshape(-1, d), yy)))


def linear_metrics(model, ys, forward_model, x_pred_sets, x_true_sets, epsilon=1e-10, xlim=(-3.5, 3.5), nbins=75, *,
                   mmd_bandwidths=None, ksd_scales=None):
    """The per-observation table of main_diffusion_linear.py:53-137 for GIVEN sample sets: x_pred_sets, x_true_sets of
    shape (n_repeats, n_obs, n, 2) (iterables of (n_obs, n, 2) CUDA tensors).  This is the part of `evaluate` that is
    arithmetic — pinned against the reference's own lines in tests/golden/eval_linear.npz.  `mmd_bandwidths`,
    `ksd_scales`: see the module docstring."""
    dev = next(model.sde.a.parameters()).device
    ys = torch.as_tensor(ys, dtype=torch.float32, device=dev).reshape(-1, model.ydim)
    n_obs = ys.shape[0]
    mean = forward_model.posterior_mean(ys)                                       # (n_obs, 2)
    cov = forward_model.posterior_cov().to(dev)
    posterior = torch.distributions.MultivariateNormal(mean[:, None, :], cov)      # batch over observations
    accs = [metrics.HistogramKL((nbins, nbins), (xlim, xlim), epsilon) for _ in range(n_obs)]
    nll_true = torch.zeros(n_obs, device=dev)
    nll_diff = torch.zeros(n_obs, device=dev)
    mse = torch.zeros(n_obs, device=dev)
    mmd = None if mmd_bandwidths is None else _MixtureMMD(mmd_bandwidths)
    ksd = None if ksd_scales is None else _SteinKSD(ksd_scales, forward_model.score_posterior)
    n_repeats = 0
    for x_pred, x_true in zip(x_pred_sets, x_true_sets):
        x_pred = torch.as_tensor(x_pred, dtype=torch.float32, device=dev)
        x_true = torch.as_tensor(x_true, dtype=torch.float32, device=dev)
        if mmd is not None:
            mmd.add(x_true, x_pred)
        score_predict, flat, yy = _score_mse(model, x_true, ys)
        score_true = forward_model.score_posterior(flat, yy)
        if ksd is not None:
            ksd.add(x_true, score_true, x_pred, ys)
        mse += ((score_predict - score_true) ** 2).sum(1).view(n_obs, -1).mean(1)
        for i in range(n_obs):
            accs[i].add(x_true[i], x_pred[i])
        nll_true -= posterior.log_prob(x_true.permute(1, 0, 2)[:, :, None, :])[:, :, 0].mean(0)
        nll_diff -= posterior.log_prob(x_pred.permute(1, 0, 2)[:, :, None, :])[:, :, 0].mean(0)
        n_repeats += 1
    table = {'KL2': np.array([a.kl() for a in accs]),
             'NLL_true': (nll_true / n_repeats).cpu().numpy(),
             'NLL_diffusion': (nll_diff / n_repeats).cpu().numpy(),
             'MSE': (mse / n_repeats).cpu().numpy()}
    if mmd is not None:
        table['MMD'] = mmd.mean()
    if ksd is not None:
        table['KSD_true'] = ksd.true.mean()
        table['KSD_diffusion'] = ksd.model.mean()
    return table


def evaluate_linear(model, ys, forward_model, out_dir=None, n_samples_x=5000, n_repeats=10, epsilon=1e-10,
                    xlim=(-3.5, 3.5), nbins=75, num_steps=200, *, mmd_bandwidths=None, ksd_scales=None):
    """`evaluate` of main_diffusion_linear.py:53-137.  ys (n_obs, 2); forward_model: dmip.linear_problem
    .LinearForwardProblem.  Returns (mean KL2, mean |NLL_true - NLL_diffusion|, mean score MSE, table); the table has an
    'MMD' column when `mmd_bandwidths` is given and 'KSD_true' / 'KSD_diffusion' columns when `ksd_scales` is given."""
    model.sde.eval()
    dev = next(model.sde.a.parameters()).device
    ys = torch.as_tensor(ys, dtype=torch.float32, device=dev).reshape(-1, model.ydim)
    mean = forward_model.posterior_mean(ys)
    posterior = torch.distributions.MultivariateNormal(mean[:, None, :], forward_model.posterior_cov().to(dev))

    def pred_sets():
        for _ in range(n_repeats):
            yield model(ys, num_samples=n_samples_x, num_steps=num_steps, return_tensor=True)   # (n_obs, n, 2)

    def true_sets():
        for _ in range(n_repeats):
            yield posterior.sample((n_samples_x,))[:, :, 0, :].permute(1, 0, 2).contiguous()   # (n_obs, n, 2)

    table = linear_metrics(model, ys, forward_model, pred_sets(), true_sets(), epsilon, xlim, nbins,
                           mmd_bandwidths=mmd_bandwidths, ksd_scales=ksd_scales)
    nlpd = np.abs(table['NLL_true'] - table['NLL_diffusion'])
    return table['KL2'].mean(), nlpd.mean(), table['MSE'].mean(), _finish(table, out_dir)


def scatterometry_metrics(model, ys, forward_model, x_pred_sets, x_true_sets, score_posterior, a, b, lambd_bd,
                          epsilon=1e-10, xlim=(-1.2, 1.2), nbins=75, *, mmd_bandwidths=None, ksd_scales=None):
    """The per-observation table of main_diffusion_scatterometry.py:40-124 for GIVEN sample sets (n_repeats, n_obs, n, 3);
    pinned against the reference's own lines in tests/golden/eval_scat.npz.  `mmd_bandwidths`, `ksd_scales`: see the module
    docstring; the model samples' KSD costs one more `score_posterior` call per repeat."""
    dev = next(model.sde.a.parameters()).device if hasattr(model.sde.a, 'parameters') else torch.device('cuda')
    ys = torch.as_tensor(ys, dtype=torch.float32, device=dev).reshape(-1, model.ydim)
    n_obs = ys.shape[0]
    rng = (xlim, xlim, xlim)
    accs = [metrics.HistogramKL((nbins,) * 3, rng, epsilon) for _ in range(n_obs)]
    nll_mcmc = torch.zeros(n_obs, device=dev)
    nll_diff = torch.zeros(n_obs, device=dev)
    mse = torch.zeros(n_obs, device=dev)
    mmd = None if mmd_bandwidths is None else _MixtureMMD(mmd_bandwidths)
    ksd = None if ksd_scales is None else _SteinKSD(ksd_scales, score_posterior)
    n_repeats = 0
    for x_pred, x_true in zip(x_pred_sets, x_true_sets):
        x_pred = torch.as_tensor(x_pred, dtype=torch.float32, device=dev)
        x_true = torch.as_tensor(x_true, dtype=torch.float32, device=dev)
        if mmd is not None:
            mmd.add(x_true, x_pred)
        n = x_true.shape[1]
        if hasattr(model.sde.a, 'prior_net'):                                                  # DPS: a = g (s_prior + s_lik)
            flat = x_true.reshape(-1, x_true.shape[-1])
            yy = ys[:, None, :].expand(n_obs, n, ys.shape[1]).reshape(flat.shape[0], -1)
            t0 = torch.zeros(flat.shape[0], 1, device=dev)
            with torch.no_grad():
                score_predict = model.sde.a(flat, yy, t0) / model.sde.base_sde.g(t0, flat)
        else:
            score_predict, flat, yy = _score_mse(model, x_true, ys)
        score_true = score_posterior(flat, yy)
        if ksd is not None:
            ksd.add(x_true, score_true, x_pred, ys)
        mse += ((score_predict - score_true) ** 2).sum(1).view(n_obs, -1).mean(1)
        for i in range(n_obs):
            accs[i].add(x_true[i], x_pred[i])
        nll_mcmc += get_log_posterior(flat, forward_model, a, b, yy, lambd_bd).view(n_obs, -1).mean(1)
        nll_diff += get_log_posterior(x_pred.reshape(-1, 3), forward_model, a, b, yy, lambd_bd).view(n_obs, -1).mean(1)
        n_repeats += 1
    table = {'KL2': np.array([acc.kl() for acc in accs]),
             'KL_reverse': np.array([acc.kl(reverse=True) for acc in accs]),
             'NLL_mcmc': (nll_mcmc / n_repeats).cpu().numpy(),
             'NLL_diffusion': (nll_diff / n_repeats).cpu().numpy(),
             'MSE': (mse / n_repeats).cpu().numpy()}
    if mmd is not None:
        table['MMD'] = mmd.mean()
    if ksd is not None:
        table['KSD_mcmc'] = ksd.true.mean()
        table['KSD_diffusion'] = ksd.model.mean()
    return table


def evaluate_scatterometry(model, ys, forward_model, gt_samples, n_samples_x, score_posterior, a, b, lambd_bd,
                           out_dir=None, n_repeats=10, epsilon=1e-10, xlim=(-1.2, 1.2), nbins=75, num_steps=200, *,
                           mmd_bandwidths=None, ksd_scales=None):
    """`evaluate` of main_diffusion_scatterometry.py:40-124.  ys (n_obs, 23); gt_samples(i, j) -> (n_samples_x, 3)
    ground-truth (Metropolis) samples of observation i, repeat j — CUDA tensor or ndarray (upstream: the files
    data/gt_samples_scatterometry/<i>/<j>.npy, see dmip.mcmc.generate_gt_samples).  Returns (mean KL2,
    mean |NLL_diffusion - NLL_mcmc|, mean score MSE, table); the table has an 'MMD' column when `mmd_bandwidths` is
    given and 'KSD_mcmc' / 'KSD_diffusion' columns when `ksd_scales` is given."""
    model.sde.eval()
    dev = next(model.sde.a.parameters()).device if hasattr(model.sde.a, 'parameters') else torch.device('cuda')
    ys = torch.as_tensor(ys, dtype=torch.float32, device=dev).reshape(-1, model.ydim)
    n_obs = ys.shape[0]

    def pred_sets():
        for _ in range(n_repeats):
            yield model(ys, num_samples=n_samples_x, num_steps=num_steps, return_tensor=True)   # (n_obs, n, 3)

    def true_sets():
        for j in range(n_repeats):
            yield torch.stack([torch.as_tensor(gt_samples(i, j), dtype=torch.float32, device=dev) for i in range(n_obs)])

    table = scatterometry_metrics(model, ys, forward_model, pred_sets(), true_sets(), score_posterior, a, b, lambd_bd,
                                  epsilon, xlim, nbins, mmd_bandwidths=mmd_bandwidths, ksd_scales=ksd_scales)
    nlpd = np.abs(table['NLL_diffusion'] - table['NLL_mcmc'])
    return table['KL2'].mean(), nlpd.mean(), table['MSE'].mean(), _finish(table, out_dir)
