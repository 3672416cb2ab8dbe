"""TEST INFRASTRUCTURE ONLY — float64 restatement of the MMD permutation two-sample test (Gretton et al. 2012, §5) that
csrc/dmip_mmd_test.cu and dmip.metrics.mmd2_test compute, on the same label bits.  Each permuted MMD^2_u is taken from
its definition (means over the kernel sub-matrices of the relabeled sets), not from the A / B / T identity the kernel
uses; `abt_statistic` states that identity separately so the tests can check one against the other.  The product never
imports this file."""
import numpy as np


def pack_labels(first):
    """bool (..., N) -> uint32 words (..., ceil(N / 32)): bit j (word j // 32, bit j % 32) set when point j is in the
    first group."""
    first = np.asarray(first, dtype=bool)
    N = first.shape[-1]
    W = -(-N // 32)
    pad = np.zeros(first.shape[:-1] + (W * 32,), dtype=np.uint64)
    pad[..., :N] = first
    return (pad.reshape(first.shape[:-1] + (W, 32)) << np.arange(32, dtype=np.uint64)).sum(-1).astype(np.uint32)


def unpack_labels(words, N):
    """uint32 words (..., W) -> bool (..., N); bits at positions >= N are dropped."""
    w = np.asarray(words).astype(np.uint32).astype(np.uint64)
    bits = (w[..., None] >> np.arange(32, dtype=np.uint64)) & 1
    return bits.reshape(w.shape[:-1] + (-1,))[..., :N].astype(bool)


def kernel_matrix(z, sigmas):
    """float64 (N, N) mixture kernel sum_b exp(-|z_i - z_j|^2 / (2 sigma_b^2)) with the diagonal set to 0."""
    z = np.asarray(z, dtype=np.float64)
    d2 = ((z[:, None, :] - z[None, :, :]) ** 2).sum(-1)
    K = sum(np.exp(-d2 / (2.0 * float(s) ** 2)) for s in sigmas)
    np.fill_diagonal(K, 0.0)
    return K


def mmd2_u(K, first):
    """MMD^2_u of the split `first` (bool (N,)) from its definition: mean_{i != j} k over the first group, the same over
    the second, minus twice the mean over the cross pairs (K has a zero diagonal)."""
    a, b = np.flatnonzero(first), np.flatnonzero(~first)
    n, m = len(a), len(b)
    kxx = K[np.ix_(a, a)].sum() / (n * (n - 1))
    kyy = K[np.ix_(b, b)].sum() / (m * (m - 1))
    kxy = K[np.ix_(a, b)].sum() / (n * m)
    return kxx + kyy - 2.0 * kxy


def abt_statistic(K, first, n, m):
    """The same statistic through A = u'Ku, B = u'K1, T = 1'K1: Sxx = A, Sxy = B - A, Syy = T - 2B + A."""
    u = np.asarray(first, dtype=np.float64)
    Ku = K @ u
    A, B, T = u @ Ku, Ku.sum(), K.sum()
    return A / (n * (n - 1)) + (T - 2 * B + A) / (m * (m - 1)) - 2 * (B - A) / (n * m)


def permutation_statistics(x, y, sigmas, labels):
    """float64 (P + 1,): MMD^2_u of x against y, then of every label row (uint32 (P, W)); NaN for a row whose popcount is
    not n."""
    n, m = len(x), len(y)
    z = np.concatenate([np.asarray(x, np.float64), np.asarray(y, np.float64)])
    K = kernel_matrix(z, sigmas)
    first = unpack_labels(labels, n + m)
    obs = np.zeros(n + m, dtype=bool)
    obs[:n] = True
    out = [mmd2_u(K, obs)]
    for row in first:
        out.append(mmd2_u(K, row) if row.sum() == n else np.nan)
    return np.array(out)


def p_value(stat, null):
    """(1 + #{null >= stat}) / (len(null) + 1); NaN when a null statistic is NaN."""
    null = np.asarray(null, dtype=np.float64)
    if np.isnan(null).any():
        return np.nan
    return (1.0 + np.count_nonzero(null >= stat)) / (len(null) + 1.0)


def random_labels(rng, P, n, m):
    """P uniformly random splits of n + m points into n and m, packed."""
    N = n + m
    first = np.zeros((P, N), dtype=bool)
    for p in range(P):
        first[p, rng.permutation(N)[:n]] = True
    return pack_labels(first)
