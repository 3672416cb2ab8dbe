"""Checks of the MMD permutation test that need no GPU: the float64 restatement (tests/mmd_perm_oracle.py) against
oracle.mmd on relabeled sets and against the A / B / T identity the kernel uses, the label bit layout of
dmip.metrics.permutation_labels, the p-value formula, the DmipMmdTest ctypes mirror, and the argument checks of
dmip.metrics.mmd2_test that run before any device work."""
import ctypes as C

import numpy as np
import pytest
import torch

import mmd_perm_oracle as mpo
from oracle import mmd as om


def _sets(n, m, d, seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, d)).astype(np.float32)
    y = (rng.standard_normal((m, d)) * 1.2 + 0.3).astype(np.float32)
    return x, y, rng


@pytest.mark.parametrize("n,m,d,sigmas", [(2, 3, 1, [1.0]), (13, 7, 3, [0.5, 1.0, 2.0]), (40, 33, 5, [1.5]),
                                          (21, 30, 16, [1.0, 2.0, 3.0, 4.0, 5.0, 6.0, 7.0, 8.0])])
def test_permuted_statistics_equal_the_mmd_oracle_on_relabeled_sets(n, m, d, sigmas):
    x, y, rng = _sets(n, m, d, seed=n * 31 + d)
    labels = mpo.random_labels(rng, 12, n, m)
    got = mpo.permutation_statistics(x, y, sigmas, labels)
    z = np.concatenate([x, y])
    first = mpo.unpack_labels(labels, n + m)
    want = [om.mmd2_terms(x, y, sigmas)[:, 0].sum()]
    want += [om.mmd2_terms(z[f], z[~f], sigmas)[:, 0].sum() for f in first]
    np.testing.assert_allclose(got, want, rtol=1e-10, atol=1e-13)


@pytest.mark.parametrize("n,m", [(2, 3), (17, 40), (64, 64)])
def test_the_abt_identity_matches_the_definition(n, m):
    x, y, rng = _sets(n, m, 3, seed=n + m)
    K = mpo.kernel_matrix(np.concatenate([x, y]), [0.7, 1.9])
    for f in mpo.unpack_labels(mpo.random_labels(rng, 20, n, m), n + m):
        assert abs(mpo.abt_statistic(K, f, n, m) - mpo.mmd2_u(K, f)) <= 1e-12


@pytest.mark.parametrize("N", [5, 31, 32, 33, 64, 1777])
def test_label_bits_round_trip(N):
    rng = np.random.default_rng(N)
    first = rng.random((3, 4, N)) < 0.4
    words = mpo.pack_labels(first)
    assert words.shape == (3, 4, -(-N // 32)) and words.dtype == np.uint32
    assert np.array_equal(mpo.unpack_labels(words, N), first)
    # bit j of word j // 32 is point j
    assert ((words[..., 0] >> 0) & 1).astype(bool).tolist() == first[..., 0].tolist()


@pytest.mark.parametrize("n,m", [(2, 3), (30, 3), (1000, 777), (16, 16)])
def test_permutation_labels_are_packed_splits_of_n_and_m(n, m):
    from dmip import metrics
    g = torch.Generator().manual_seed(5)
    lab = metrics.permutation_labels(2, n, m, 7, generator=g, device="cpu")
    W = -(-(n + m) // 32)
    assert lab.shape == (2, 7, W) and lab.dtype == torch.int32
    words = lab.numpy().view(np.uint32)
    first = mpo.unpack_labels(words, n + m)
    assert (first.sum(-1) == n).all()
    assert np.array_equal(mpo.pack_labels(first), words)               # no bit at positions >= N
    assert len({f.tobytes() for f in first.reshape(-1, n + m)}) > 1
    again = metrics.permutation_labels(2, n, m, 7, generator=torch.Generator().manual_seed(5), device="cpu")
    assert torch.equal(lab, again)


def test_p_value_formula():
    assert mpo.p_value(1.0, [0.5, 2.0, 1.0, -3.0]) == 3 / 5           # ties count as exceedances
    assert mpo.p_value(5.0, np.zeros(254)) == 1 / 255
    assert mpo.p_value(-5.0, np.zeros(254)) == 1.0
    assert np.isnan(mpo.p_value(0.0, [1.0, np.nan]))
    x, y, rng = _sets(6, 5, 2, seed=3)
    lab = mpo.random_labels(rng, 9, 6, 5)
    lab[4, 0] ^= 1                                                       # one row with n +- 1 bits
    s = mpo.permutation_statistics(x, y, [1.0], lab)
    assert np.isnan(s[5]) and not np.isnan(np.delete(s, 5)).any()


def test_ctypes_mirror_matches_the_header():
    from dmip import metrics
    from test_abi import _sizeof_from_c
    assert C.sizeof(metrics.DmipMmdTest) == _sizeof_from_c(["DmipMmdTest"])["DmipMmdTest"]


def _labels(n_obs, n, m, P, dtype=torch.int32):
    return torch.zeros(n_obs, P, -(-(n + m) // 32), dtype=dtype)


@pytest.mark.parametrize("kw", [
    dict(x=(10, 3), y=(12, 2)),                 # dimensions differ
    dict(x=(10, 17), y=(12, 17)),               # d > 16
    dict(x=(1, 3), y=(12, 3)),                  # n < 2
    dict(x=(10, 3), y=(1, 3)),                  # m < 2
    dict(x=(2, 10, 3), y=(3, 12, 3)),           # observation counts differ
    dict(x=(10, 3), y=(2, 12, 3)),              # batched and unbatched mixed
    dict(bw=[]), dict(bw=[1.0] * 9), dict(bw=[0.0]), dict(bw=[-1.0]), dict(bw=[float("nan")]), dict(bw=[float("inf")]),
    dict(P=0), dict(P=-3), dict(P=2.5), dict(P=True),
    dict(x=(600000, 3), y=(600000, 3)),         # n + m > 2^20
])
def test_mmd2_test_rejects_invalid_arguments_before_touching_a_device(kw):
    from dmip import metrics
    x = torch.zeros(kw.get("x", (10, 3)))
    y = torch.zeros(kw.get("y", (12, 3)))
    with pytest.raises(ValueError):
        metrics.mmd2_test(x, y, kw.get("bw", [1.0]), kw.get("P", 254))


@pytest.mark.parametrize("labels", [
    _labels(1, 10, 12, 0),                      # no permutation
    _labels(1, 10, 12, 255),                    # more than one call takes
    _labels(2, 10, 12, 4),                      # observation count differs
    torch.zeros(1, 4, 2, dtype=torch.int32),    # wrong word count (22 points need 1)
    torch.zeros(4, 1, dtype=torch.int32),       # not 3-D
    _labels(1, 10, 12, 4, dtype=torch.int64),   # not 32-bit words
])
def test_permutation_statistics_reject_bad_labels_before_touching_a_device(labels):
    from dmip import metrics
    with pytest.raises(ValueError):
        metrics.mmd2_permutation_statistics(torch.zeros(10, 3), torch.zeros(12, 3), [1.0], labels)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU refusal path")
def test_mmd2_test_has_no_cpu_fallback():
    from dmip import metrics
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        metrics.mmd2_test(torch.zeros(10, 3), torch.zeros(12, 3), [1.0])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        metrics.mmd2_permutation_statistics(torch.zeros(10, 3), torch.zeros(12, 3), [1.0], _labels(1, 10, 12, 3))
