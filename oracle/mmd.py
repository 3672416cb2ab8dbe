"""TEST INFRASTRUCTURE ONLY — float64 restatement of the unbiased MMD^2 of Gretton et al. 2012 (JMLR 13, eq. 3) with Gaussian kernels
k(a, b) = exp(-|a - b|^2 / (2 sigma^2)), and the closed forms of its kernel means for isotropic Gaussians.  The
product (csrc/dmip_mmd.cu, dmip.metrics.mmd2) never imports it.  The reference has no MMD, so
this is the whole oracle (parity unpinned)."""
import numpy as np


def _kernel_sums(a, b, sigmas, exclude_diagonal, chunk_pairs=1 << 22):
    """sum_{i,j} k_s(a_i, b_j) for every sigma s, in float64, over row chunks; exclude_diagonal drops i == j (a is b)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    inv = np.array([-0.5 / float(s) ** 2 for s in sigmas])
    rows = max(1, chunk_pairs // max(1, b.shape[0]))
    out = np.zeros(len(sigmas))
    bb = (b * b).sum(1)
    for r0 in range(0, a.shape[0], rows):
        ac = a[r0:r0 + rows]
        # |a|^2 + |b|^2 - 2 a.b in float64: the cancellation error (~1e-16 |a|^2) is far below the fp32 inputs' rounding
        d2 = np.maximum((ac * ac).sum(1)[:, None] + bb[None, :] - 2.0 * (ac @ b.T), 0.0)
        if exclude_diagonal:
            i = np.arange(r0, min(r0 + rows, a.shape[0]))
            d2[i - r0, i] = np.inf
        for k, c in enumerate(inv):
            out[k] += np.exp(c * d2).sum()
    return out


def mmd2_terms(x, y, sigmas):
    """(n_bw, 4) float64 array {MMD^2_u, Kxx, Kyy, Kxy} for samples x (n, d), y (m, d)."""
    n, m = len(x), len(y)
    kxx = _kernel_sums(x, x, sigmas, True) / (n * (n - 1))
    kyy = _kernel_sums(y, y, sigmas, True) / (m * (m - 1))
    kxy = _kernel_sums(x, y, sigmas, False) / (n * m)
    return np.stack([kxx + kyy - 2 * kxy, kxx, kyy, kxy], axis=-1)


def mmd2_terms_naive(x, y, sigmas):
    """The same estimator as an explicit O(n^2) double loop (checks mmd2_terms on small inputs)."""
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    n, m = len(x), len(y)
    out = []
    for s in sigmas:
        k = lambda a, b: np.exp(-np.sum((a - b) ** 2) / (2.0 * s * s))
        kxx = sum(k(x[i], x[j]) for i in range(n) for j in range(n) if i != j) / (n * (n - 1))
        kyy = sum(k(y[i], y[j]) for i in range(m) for j in range(m) if i != j) / (m * (m - 1))
        kxy = sum(k(x[i], y[j]) for i in range(n) for j in range(m)) / (n * m)
        out.append([kxx + kyy - 2 * kxy, kxx, kyy, kxy])
    return np.array(out)


def gaussian_kernel_mean(sigma, d, s1, s2, mu_diff=0.0):
    """E k(X, Y) for independent X ~ N(mu_1, s1^2 I_d), Y ~ N(mu_2, s2^2 I_d), |mu_1 - mu_2| = mu_diff:
    (sigma^2 / (sigma^2 + s1^2 + s2^2))^(d/2) exp(-mu_diff^2 / (2 (sigma^2 + s1^2 + s2^2)))."""
    v = sigma ** 2 + s1 ** 2 + s2 ** 2
    return (sigma ** 2 / v) ** (d / 2) * np.exp(-mu_diff ** 2 / (2 * v))


def population_terms(sigma, d, s1, s2, mu_diff):
    """{MMD^2, E k(X,X'), E k(Y,Y'), E k(X,Y)} for X ~ N(mu_1, s1^2 I), Y ~ N(mu_2, s2^2 I)."""
    kxx = gaussian_kernel_mean(sigma, d, s1, s1)
    kyy = gaussian_kernel_mean(sigma, d, s2, s2)
    kxy = gaussian_kernel_mean(sigma, d, s1, s2, mu_diff)
    return np.array([kxx + kyy - 2 * kxy, kxx, kyy, kxy])
