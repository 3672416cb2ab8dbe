"""MMD^2 checks that need no GPU: the float64 oracle (oracle/mmd.py) against a naive double loop and against the closed
forms of Gaussian kernel means, the DmipMmd ctypes mirror against the C header, and the argument checks of
dmip.metrics.mmd2 that run before any device work."""
import numpy as np
import pytest
import torch

from oracle import mmd as om


@pytest.mark.parametrize("n,m,d", [(2, 3, 1), (7, 5, 3), (30, 17, 16)])
def test_oracle_matches_the_naive_double_loop(n, m, d):
    rng = np.random.default_rng(n * 100 + d)
    x = rng.standard_normal((n, d)).astype(np.float32)
    y = (rng.standard_normal((m, d)) * 1.3 + 0.2).astype(np.float32)
    sig = [0.5 * d ** 0.5, d ** 0.5, 3.0]
    np.testing.assert_allclose(om.mmd2_terms(x, y, sig), om.mmd2_terms_naive(x, y, sig), rtol=1e-12, atol=1e-14)


def test_oracle_means_match_the_closed_forms():
    """N(0, I) against N((0.05, 0), I) in d = 2, sigma = 1, 20 000 samples each.  Population values: Kxx = Kyy = 1/3,
    Kxy = 0.333194, MMD^2 = 2.7772e-4.  Bars are 4 standard deviations of the U-statistics at this n (Kxx: sqrt(4 Var
    E[k(x, X') | x] / n) = 1.7e-3; MMD^2_u: sqrt(8 * 3.9e-5 / n) = 1.25e-4)."""
    rng = np.random.default_rng(0)
    n = 20000
    x = rng.standard_normal((n, 2))
    y = rng.standard_normal((n, 2)) + np.array([0.05, 0.0])
    got = om.mmd2_terms(x, y, [1.0])[0]
    want = om.population_terms(1.0, 2, 1.0, 1.0, 0.05)
    np.testing.assert_allclose(want, [2.7772e-4, 1 / 3, 1 / 3, 0.333194], rtol=2e-5)
    assert np.all(np.abs(got[1:] - want[1:]) <= 7e-3), (got, want)
    assert abs(got[0] - want[0]) <= 5e-4, (got, want)


def test_ctypes_mirror_matches_the_header():
    from dmip import metrics
    from test_abi import _sizeof_from_c
    import ctypes as C
    assert C.sizeof(metrics.DmipMmd) == _sizeof_from_c(["DmipMmd"])["DmipMmd"]


@pytest.mark.parametrize("x,y,bw", [
    ((10, 3), (12, 2), [1.0]),          # dimensions differ
    ((10, 17), (12, 17), [1.0]),        # d > 16
    ((1, 3), (12, 3), [1.0]),           # n < 2
    ((10, 3), (1, 3), [1.0]),           # m < 2
    ((2, 10, 3), (3, 12, 3), [1.0]),    # observation counts differ
    ((10, 3), (2, 12, 3), [1.0]),       # batched and unbatched mixed
    ((10,), (12,), [1.0]),              # not (n, d)
    ((10, 3), (12, 3), []),             # no bandwidth
    ((10, 3), (12, 3), [1.0] * 9),      # more than 8
    ((10, 3), (12, 3), [0.0]),
    ((10, 3), (12, 3), [-1.0]),
    ((10, 3), (12, 3), [float("nan")]),
    ((10, 3), (12, 3), [float("inf")]),
])
def test_mmd2_rejects_invalid_arguments_before_touching_a_device(x, y, bw):
    from dmip import metrics
    with pytest.raises(ValueError):
        metrics.mmd2(torch.zeros(x), torch.zeros(y), bw)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU refusal path")
def test_mmd2_has_no_cpu_fallback():
    from dmip import metrics
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        metrics.mmd2(torch.zeros(10, 3), torch.zeros(12, 3), [1.0])
