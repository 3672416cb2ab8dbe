"""Kernel Stein discrepancy checks that need no GPU: the float64 oracle (oracle/ksd.py) against a naive double loop, against
torch float64 autograd of the Stein kernel's definition and, by Monte Carlo, against the Gaussian closed form; the
DmipKsd ctypes mirror against the C header; and the argument checks of dmip.metrics.ksd2 that run before any device
work."""
import numpy as np
import pytest
import torch

from oracle import ksd as ok

KERNELS = ["imq", "gaussian"]


def _sample(n, d, seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, d)) * 0.8 + 0.1
    s = -x * 1.3 + 0.2 * rng.standard_normal((n, d))   # a score that is not that of x's own law
    return x, s


@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("n,d", [(2, 1), (9, 3), (13, 16)])
def test_oracle_matches_the_naive_double_loop(kernel, n, d):
    x, s = _sample(n, d, n * 100 + d)
    sc = [0.5 * d ** 0.5, d ** 0.5, 3.0]
    np.testing.assert_allclose(ok.ksd2_terms(x, s, sc, kernel), ok.ksd2_terms_naive(x, s, sc, kernel), rtol=1e-12,
                               atol=1e-14)


def _stein_autograd(kfun, x, xp, s, sp):
    """u(x, x') = s.s' k + s.grad_x' k + s'.grad_x k + tr grad_x grad_x' k through torch float64 autograd."""
    x = x.clone().requires_grad_(True)
    xp = xp.clone().requires_grad_(True)
    k = kfun(x, xp)
    gx, gxp = torch.autograd.grad(k, (x, xp), create_graph=True)
    tr = sum(torch.autograd.grad(gx[a], xp, retain_graph=True)[0][a] for a in range(x.numel()))
    return ((s @ sp) * k + s @ gxp + sp @ gx + tr).detach()


@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("d", [1, 3, 16])
def test_oracle_matches_autograd_of_the_stein_kernel_definition(kernel, d):
    n, c = 6, 1.3
    x, s = _sample(n, d, 7 * d)
    if kernel == "imq":
        kfun = lambda a, b: (c * c + ((a - b) ** 2).sum()) ** -0.5
    else:
        kfun = lambda a, b: torch.exp(-((a - b) ** 2).sum() / (2 * c * c))
    X, S = torch.from_numpy(x), torch.from_numpy(s)
    u = torch.stack([torch.stack([_stein_autograd(kfun, X[i], X[j], S[i], S[j]) for j in range(n)])
                     for i in range(n)]).numpy()
    off = u.sum() - np.trace(u)
    want = np.array([off / (n * (n - 1)), u.sum() / (n * n)])
    np.testing.assert_allclose(ok.ksd2_terms(x, s, [c], kernel)[0], want, rtol=1e-12, atol=1e-14)


def test_gaussian_closed_form_is_the_population_value():
    """p = N(0, I_2), samples N((0.4, 0.4), I_2), sigma = 0.8: KSD^2 = |m|^2 (1 + 2 / sigma^2)^(-d/2) = 0.077576.  The
    U-statistic is unbiased, so the mean over 30 independent sets of 1500 meets it within 4 standard errors (the standard
    error is estimated from the same 30 values)."""
    m, sigma = np.array([0.4, 0.4]), 0.8
    pop = ok.gaussian_shift_ksd2(m, sigma)
    assert abs(pop - 0.077576) < 1e-6
    rng = np.random.default_rng(0)
    vals = []
    for _ in range(30):
        x = rng.standard_normal((1500, 2)) + m
        vals.append(ok.ksd2_terms(x, -x, [sigma], "gaussian")[0, 0])
    vals = np.array(vals)
    se = vals.std(ddof=1) / np.sqrt(len(vals))
    assert abs(vals.mean() - pop) <= 4 * se, (vals.mean(), se, pop)


def test_ctypes_mirror_matches_the_header():
    from dmip import metrics
    from test_abi import _sizeof_from_c
    import ctypes as C
    assert C.sizeof(metrics.DmipKsd) == _sizeof_from_c(["DmipKsd"])["DmipKsd"]


@pytest.mark.parametrize("x,s,sc,kernel", [
    ((10, 3), (10, 2), [1.0], "imq"),          # shapes differ
    ((10, 3), (12, 3), [1.0], "imq"),          # sample counts differ
    ((2, 10, 3), (3, 10, 3), [1.0], "imq"),    # observation counts differ
    ((10, 3), (1, 10, 3), [1.0], "imq"),       # batched and unbatched mixed
    ((10, 17), (10, 17), [1.0], "imq"),        # d > 16
    ((1, 3), (1, 3), [1.0], "imq"),            # n < 2
    ((2, 1, 3), (2, 1, 3), [1.0], "gaussian"),  # n < 2, batched
    ((0, 10, 3), (0, 10, 3), [1.0], "imq"),    # no observation
    ((10,), (10,), [1.0], "imq"),              # not (n, d)
    ((10, 3), (10, 3), [], "imq"),             # no scale
    ((10, 3), (10, 3), [1.0] * 9, "imq"),      # more than 8
    ((10, 3), (10, 3), [0.0], "imq"),
    ((10, 3), (10, 3), [-1.0], "gaussian"),
    ((10, 3), (10, 3), [float("nan")], "imq"),
    ((10, 3), (10, 3), [float("inf")], "imq"),
    ((10, 3), (10, 3), 1.0, "imq"),            # not a sequence
    ((10, 3), (10, 3), [1.0], "rbf"),          # unknown kernel
])
def test_ksd2_rejects_invalid_arguments_before_touching_a_device(x, s, sc, kernel):
    from dmip import metrics
    with pytest.raises(ValueError):
        metrics.ksd2(torch.zeros(x), torch.zeros(s), sc, kernel)


def test_ksd2_rejects_non_tensors():
    from dmip import metrics
    with pytest.raises(ValueError):
        metrics.ksd2(np.zeros((10, 3)), torch.zeros(10, 3), [1.0])


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU refusal path")
def test_ksd2_has_no_cpu_fallback():
    from dmip import metrics
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        metrics.ksd2(torch.zeros(10, 3), torch.zeros(10, 3), [1.0])
