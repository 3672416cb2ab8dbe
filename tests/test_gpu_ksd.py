"""GPU tests of the kernel Stein discrepancy kernel (csrc/dmip_ksd.cu) through dmip.metrics.ksd2 and the C ABI
(pytest -m gpu).

Bar: |KSD^2_U - oracle| and |KSD^2_V - oracle| <= 2e-6 x the oracle's mean |u_ij| (i != j) on the same fp32 inputs.  Each
pair value is fp32: its terms carry a few ulp (6e-8 each) of rounding plus the MUFU's relative error (rsqrt.approx
< 2^-22.9, ex2.approx 2 ulp), which k^5 multiplies by five: <= 1e-6 of the terms' size per pair, mostly of either sign.
Row sums are fp32 over <= 2048 pairs (a random walk of sqrt(2048) x 6e-8 = 2.7e-6 of the row's sum of |u| at worst,
averaged down over the rows) and fp64 from there on, u_ii fp64 throughout."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import ksd as ok

pytestmark = pytest.mark.gpu
DEV = "cuda"
REL_TOL = 2e-6
KERNELS = ["imq", "gaussian"]


def _sets(n_obs, n, d, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n_obs, n, d, generator=g) * 0.8 + 0.1
    s = -1.3 * x + 0.2 * torch.randn(n_obs, n, d, generator=g)
    return x, s


def _scales(ns, d):
    return [float(c) for c in np.geomspace(0.3, 3.0, ns) * d ** 0.5] if ns > 1 else [float(d ** 0.5)]


def _check(got, x, s, sc, kernel):
    """got (n_obs, n_scales, 2) against the oracle on the same fp32 values — the scales too, which the kernel receives as
    fp32 (at the smallest Gaussian scales the closed-form u_ii alone moves by 1e-4 of mean |u| between a float64 scale and
    its fp32 rounding); returns the worst error over mean |u|"""
    worst = 0.0
    sc = [float(np.float32(c)) for c in sc]
    for o in range(x.shape[0]):
        xo, so = x[o].double().numpy(), s[o].double().numpy()
        t = ok.stein_sums(xo, so, sc, kernel)
        n = xo.shape[0]
        ref = np.stack([t[:, 0] / (n * (n - 1)), (t[:, 0] + t[:, 1]) / (n * n)], axis=-1)
        scale = t[:, 2] / (n * (n - 1))
        err = np.abs(np.asarray(got[o]) - ref).max(-1) / scale
        worst = max(worst, float(err.max()))
        assert np.all(err <= REL_TOL), (o, kernel, err, got[o], ref)
    return worst


# (n, n_obs, n_scales): n in {2, 3, 127, 128, 129, 1000, 4099}, 1 and 5 observations, 1 and 8 scales; tile edges are
# 512, 1024 or 2048 rows, so 1000 crosses a tile edge in some builds and 4099 is ragged in every build of the kernel
CONFIGS = [(2, 1, 1), (3, 5, 8), (127, 5, 1), (128, 1, 8), (129, 5, 8), (1000, 1, 8), (4099, 1, 1)]


@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("d", list(range(1, 17)))
def test_ksd2_matches_the_float64_oracle(d, kernel):
    from dmip import metrics
    for k, (n, n_obs, ns) in enumerate(CONFIGS):
        x, s = _sets(n_obs, n, d, seed=100 * d + k)
        sc = _scales(ns, d)
        got = metrics.ksd2(x.to(DEV), s.to(DEV), sc, kernel, terms=True).cpu().numpy()
        assert got.shape == (n_obs, ns, 2)
        _check(got, x, s, sc, kernel)


def _scat_golden_with_scores():
    """eval_scat golden ground-truth samples (3 observations x 2000, d = 3) and their surrogate posterior scores"""
    import gpu_cases as gc
    from util import load_golden
    from dmip.utils_scatterometry import make_score_posterior
    fx = load_golden("eval_scat", dtype=torch.float64)
    x = fx["x_true"][:, 0].float().contiguous().to(DEV)               # (3, 2000, 3)
    ys = fx["ys"].float().to(DEV)
    fm, _ = gc._surrogate_module()
    sp = make_score_posterior(fm, dict(a=0.2, b=0.01, lambd_bd=1000))
    n_obs, n, d = x.shape
    yy = ys[:, None, :].expand(n_obs, n, ys.shape[1]).reshape(n_obs * n, -1)
    s = sp(x.reshape(-1, d), yy).detach().reshape(n_obs, n, d).float().contiguous()
    return x, s


@pytest.mark.parametrize("kernel", KERNELS)
def test_ksd2_matches_the_oracle_on_scatterometry_samples_with_surrogate_scores(kernel):
    from dmip import metrics
    x, s = _scat_golden_with_scores()
    assert torch.isfinite(s).all()
    sc = [0.1, 0.3, 1.0]
    got = metrics.ksd2(x, s, sc, kernel, terms=True).cpu().numpy()
    _check(got, x.cpu(), s.cpu(), sc, kernel)


def test_population_value_at_one_million_samples():
    """p = N(0, I_2), n = 2^20 samples of N((0.4, 0.4), I_2), Gaussian kernel sigma = 0.8: KSD^2_U within 5 estimator
    standard deviations of |m|^2 (1 + 2 / sigma^2)^(-1) = 0.077576.  The standard deviation, 3.2e-4, is scaled from the
    spread of 60 float64 sets of 1500 (0.0085 each) by sqrt(1500 / 2^20)."""
    from dmip import metrics
    g = torch.Generator(device=DEV).manual_seed(2026)
    m = torch.tensor([0.4, 0.4], device=DEV)
    x = torch.randn(1 << 20, 2, device=DEV, generator=g) + m
    got = metrics.ksd2(x, -x, [0.8], "gaussian", terms=True)[0].cpu().numpy()
    pop = ok.gaussian_shift_ksd2([0.4, 0.4], 0.8)
    assert abs(got[0] - pop) <= 5 * 3.2e-4, (got, pop)
    assert got[1] >= got[0] - 1e-6


def _linear_posterior(y, n_obs, n, seed):
    from dmip.linear_problem import LinearForwardProblem
    fp = LinearForwardProblem()
    ys = torch.as_tensor(y, dtype=torch.float32, device=DEV)
    mean = fp.posterior_mean(ys).to(DEV)
    cov = fp.posterior_cov().to(DEV)
    torch.manual_seed(seed)
    x = torch.distributions.MultivariateNormal(mean, cov).sample((n_obs, n)).float()
    return fp, ys, x, cov


def test_null_and_alternative_on_the_linear_posterior():
    """Exact posterior samples: 16 sets of 2^14 give IMQ KSD^2_U consistent with 0 (|mean| <= 4 standard errors).  The
    same posterior sampled at 2^18 and shifted by 0.1 posterior standard deviations per coordinate is clearly positive
    (above 10 null standard deviations of the smaller sets).  V >= 0 throughout."""
    from dmip import metrics
    y = [0.4, -0.7]
    fp, ys, x, cov = _linear_posterior(y, 16, 1 << 14, seed=3)
    score = fp.score_posterior(x.reshape(-1, 2), ys.expand(x.shape[0] * x.shape[1], 2)).reshape(x.shape)
    null = metrics.ksd2(x, score, [1.0], terms=True)[:, 0].cpu().numpy()      # (16, 2)
    se = null[:, 0].std(ddof=1) / np.sqrt(len(null))
    assert abs(null[:, 0].mean()) <= 4 * se, (null[:, 0].mean(), se)
    assert np.all(null[:, 1] >= 0), null
    _, _, xa, _ = _linear_posterior(y, 1, 1 << 18, seed=4)
    xa = (xa[0] + 0.1 * cov.diagonal().sqrt()).contiguous()
    sa = fp.score_posterior(xa, ys.expand(xa.shape[0], 2))
    alt = metrics.ksd2(xa, sa, [1.0], terms=True)[0].cpu().numpy()
    assert alt[0] > 10 * null[:, 0].std(ddof=1) and alt[1] >= 0, (alt, null[:, 0].std(ddof=1))


def test_determinism_batching_launches_and_nan_scores():
    from dmip import _lib, metrics
    x, s = _sets(5, 3000, 3, seed=11)
    x, s = x.to(DEV), s.to(DEV)
    sc = [0.7, 1.5, 3.0]
    for kernel in KERNELS:
        a = metrics.ksd2(x, s, sc, kernel, terms=True)
        assert _lib.lib().dmip_last_launch_count() <= 2
        b = metrics.ksd2(x, s, sc, kernel, terms=True)
        assert torch.equal(a, b), "two calls differ"
        for o in range(5):
            single = metrics.ksd2(x[o], s[o], sc, kernel, terms=True)
            scale = ok.mean_abs_u(x[o].double().cpu().numpy(), s[o].double().cpu().numpy(), sc, kernel)
            assert ((single - a[o]).abs().cpu().numpy().max(-1) <= REL_TOL * scale).all(), o
        assert metrics.ksd2(x[0], s[0], sc, kernel).shape == (3,) and metrics.ksd2(x, s, sc, kernel).shape == (5, 3)
    s_bad = s.clone()
    s_bad[2, 17, 1] = float("inf")
    got = metrics.ksd2(x, s_bad, sc, terms=True)
    assert torch.isnan(got[2]).all() and torch.isfinite(got[[0, 1, 3, 4]]).all()


def test_guarded_buffers_and_invalid_arguments():
    from dmip import metrics
    os.environ["DMIP_GUARD"] = "1"
    try:
        for kernel in KERNELS:
            for (n, n_obs, d, ns) in [(2, 1, 1, 1), (1027, 3, 3, 8), (2049, 2, 2, 5), (515, 4, 16, 2), (1025, 2, 7, 6),
                                      (4099, 1, 4, 8)]:
                x, s = _sets(n_obs, n, d, seed=n + d)
                metrics.ksd2(x.to(DEV), s.to(DEV), _scales(ns, d), kernel, terms=True)   # raises on a canary hit
    finally:
        os.environ.pop("DMIP_GUARD", None)
    x, s = torch.zeros(10, 3, device=DEV), torch.zeros(10, 3, device=DEV)
    for bad in ([], [1.0] * 9, [0.0], [-1.0], [float("nan")], [float("inf")]):
        with pytest.raises(ValueError):
            metrics.ksd2(x, s, bad)
    with pytest.raises(ValueError):
        metrics.ksd2(x, s[:9], [1.0])
    # the C entry point checks the same conditions itself
    L = metrics._bind()
    out = torch.empty(64, dtype=torch.float64, device=DEV)
    keep = []

    def desc(**kw):
        d = metrics.DmipKsd()
        d.dim, d.n_obs, d.n, d.kernel, d.n_scales = 3, 1, 10, 0, 1
        d.scale[0] = 1.0
        d.x, d.score, d.out = x.data_ptr(), s.data_ptr(), out.data_ptr()
        for k, v in kw.items():
            if k == "scale":
                d.scale[0] = v
            else:
                setattr(d, k, v)
        nbytes = L.dmip_ksd_workspace_bytes(C.byref(d))
        ws = torch.empty(max(nbytes, 8) + 8, dtype=torch.uint8, device=DEV)
        keep.append(ws)
        d.workspace, d.workspace_bytes = ws.data_ptr(), nbytes
        return d

    for kw in (dict(dim=0), dict(dim=17), dict(n_obs=0), dict(n=1), dict(kernel=2), dict(kernel=-1), dict(n_scales=0),
               dict(n_scales=9), dict(scale=0.0), dict(scale=-2.0), dict(scale=float("inf")), dict(scale=float("nan")),
               dict(x=None), dict(score=None), dict(out=None)):
        rc = L.dmip_ksd(C.byref(desc(**kw)), None)
        assert rc == -1 and L.dmip_last_error(), (kw, rc)
    d = desc()
    d.workspace += 4
    assert L.dmip_ksd(C.byref(d), None) == -1 and b"aligned" in L.dmip_last_error()
    d = desc()
    d.workspace_bytes -= 8
    assert L.dmip_ksd(C.byref(d), None) == -3 and b"workspace" in L.dmip_last_error()
    d = desc()
    d.workspace = None
    assert L.dmip_ksd(C.byref(d), None) == -3
    assert L.dmip_ksd_workspace_bytes(C.byref(desc(n_obs=3, n_scales=2))) == (1024 + 3) * 2 * 2 * 8
    assert L.dmip_ksd_workspace_bytes(C.byref(desc(n=1 << 30, n_obs=3, n_scales=2))) == (1024 + 3) * 2 * 2 * 8
    assert L.dmip_ksd(C.byref(desc()), None) == 0
    torch.cuda.synchronize()


def _eval_tables(problem, ksd_scales):
    import gpu_cases as gc
    from util import load_golden
    from dmip import evaluation
    from dmip.linear_problem import LinearForwardProblem
    from dmip.models.diffusion import CDE
    from dmip.utils_scatterometry import make_score_posterior
    from oracle.weights import make_params, state_dict_from_params
    fx = load_golden("eval_" + problem, dtype=torch.float64)
    xp, xt = fx["x_pred"].float(), fx["x_true"].float()
    sets = lambda v: [v[:, j].contiguous().to(DEV) for j in range(v.shape[1])]
    kw = {} if ksd_scales == "absent" else dict(ksd_scales=ksd_scales)
    ys = fx["ys"].float()
    if problem == "linear":
        m = gc.trained_model()
        m.sde.a.precision = "fp32"
        fp = LinearForwardProblem()
        score = fp.score_posterior
        table = evaluation.linear_metrics(m, ys, fp, sets(xp), sets(xt), **kw)
    else:
        fm, _ = gc._surrogate_module()
        m = CDE(3, 23, [512, 512, 512])
        m.sde.a.load_state_dict(state_dict_from_params(make_params(95, 27, 3)))
        m.sde.to(DEV)
        m.sde.a.precision = "fp32"
        score = make_score_posterior(fm, dict(a=0.2, b=0.01, lambd_bd=1000))
        table = evaluation.scatterometry_metrics(m, ys, fm, sets(xp), sets(xt), score, 0.2, 0.01, 1000, **kw)
    return table, xp, xt, ys.to(DEV), score


@pytest.mark.parametrize("problem", ["linear", "scat"])
def test_evaluate_tables_with_and_without_ksd(problem):
    from dmip import metrics
    base, xp, xt, ys, score = _eval_tables(problem, "absent")
    none = _eval_tables(problem, None)[0]
    assert list(none) == list(base) and not any(k.startswith("KSD") for k in none)
    for k in base:
        assert np.array_equal(none[k], base[k]), k
    sc = (0.25, 0.5, 1.0)
    with_ksd = _eval_tables(problem, sc)[0]
    truth = "KSD_true" if problem == "linear" else "KSD_mcmc"
    assert list(with_ksd) == list(base) + [truth, "KSD_diffusion"]
    for k in base:
        assert np.array_equal(with_ksd[k], base[k]), k
    n_obs, n_rep, n, d = xp.shape
    yy = ys[:, None, :].expand(n_obs, n, ys.shape[1]).reshape(n_obs * n, -1)

    def direct(v):
        vals = []
        for j in range(n_rep):
            x = v[:, j].contiguous().to(DEV)
            s = score(x.reshape(-1, d), yy).reshape(x.shape)
            vals.append(metrics.ksd2(x, s, sc).sum(-1).cpu().numpy())
        return np.mean(vals, axis=0)

    for col, v in ((truth, xt), ("KSD_diffusion", xp)):
        ref = direct(v)
        assert np.allclose(with_ksd[col], ref, rtol=1e-12, atol=0), (col, with_ksd[col], ref)
