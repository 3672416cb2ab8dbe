"""TEST INFRASTRUCTURE ONLY — float64 restatement of the kernel Stein discrepancy (Liu, Lee & Jordan 2016; Chwialkowski,
Strathmann & Gretton 2016) of samples x_i with target scores s_i = grad log p(x_i), for the IMQ kernel
k = (c^2 + r^2)^(-1/2) and the Gaussian kernel k = exp(-r^2 / (2 sigma^2)).  With delta = x_i - x_j, r^2 = |delta|^2,
a = (s_i - s_j).delta + d:
    IMQ:      u_ij = k s_i.s_j + k^3 a - 3 r^2 k^5,          u_ii = |s_i|^2 / c + d / c^3
    Gaussian: u_ij = k [s_i.s_j + a / sigma^2 - r^2 / sigma^4], u_ii = |s_i|^2 + d / sigma^2
KSD^2_U = sum_{i != j} u_ij / (n (n - 1)),  KSD^2_V = sum_{i, j} u_ij / n^2.  The product (csrc/dmip_ksd.cu,
dmip.metrics.ksd2) never imports it.  The reference has no KSD, so this is the whole oracle (parity unpinned)."""
import numpy as np


def _u(kernel, scale, d, r2, ss, a):
    """Stein kernel values from r^2, s_i.s_j and a = (s_i - s_j).delta + d (float64 arrays of one shape)."""
    if kernel == "imq":
        k = 1.0 / np.sqrt(scale * scale + r2)
        return k * ss + k ** 3 * a - 3.0 * r2 * k ** 5
    if kernel == "gaussian":
        s2 = scale * scale
        return np.exp(-r2 / (2.0 * s2)) * (ss + a / s2 - r2 / (s2 * s2))
    raise ValueError(kernel)


def stein_sums(x, s, scales, kernel, chunk_pairs=1 << 18):
    """(n_scales, 3) float64: {sum_{i != j} u_ij, sum_i u_ii, sum_{i != j} |u_ij|} over row chunks, direct differences."""
    x = np.asarray(x, dtype=np.float64)
    s = np.asarray(s, dtype=np.float64)
    n, d = x.shape
    rows = max(1, chunk_pairs // max(1, n))
    out = np.zeros((len(scales), 3))
    for r0 in range(0, n, rows):
        xa, sa = x[r0:r0 + rows], s[r0:r0 + rows]
        delta = xa[:, None, :] - x[None, :, :]
        r2 = np.einsum("ijk,ijk->ij", delta, delta)
        ss = sa @ s.T
        a = np.einsum("ijk,ijk->ij", sa[:, None, :] - s[None, :, :], delta) + d
        off = np.ones(r2.shape, dtype=bool)
        i = np.arange(r0, r0 + xa.shape[0])
        off[i - r0, i] = False
        for b, c in enumerate(scales):
            u = _u(kernel, float(c), d, r2, ss, a)
            out[b, 0] += u[off].sum()
            out[b, 2] += np.abs(u[off]).sum()
    q = (s * s).sum(1)
    for b, c in enumerate(scales):
        c = float(c)
        out[b, 1] = (q / c + d / c ** 3).sum() if kernel == "imq" else (q + d / (c * c)).sum()
    return out


def ksd2_terms(x, s, scales, kernel="imq"):
    """(n_scales, 2) float64 {KSD^2_U, KSD^2_V} for samples x (n, d) with scores s (n, d)."""
    n = len(x)
    t = stein_sums(x, s, scales, kernel)
    return np.stack([t[:, 0] / (n * (n - 1)), (t[:, 0] + t[:, 1]) / (n * n)], axis=-1)


def mean_abs_u(x, s, scales, kernel="imq"):
    """(n_scales,) mean_{i != j} |u_ij|: the scale the device results' fp32 error is measured on."""
    n = len(x)
    return stein_sums(x, s, scales, kernel)[:, 2] / (n * (n - 1))


def ksd2_terms_naive(x, s, scales, kernel="imq"):
    """The same estimator as an explicit O(n^2) double loop over the table's formulas (checks ksd2_terms)."""
    x = np.asarray(x, dtype=np.float64)
    s = np.asarray(s, dtype=np.float64)
    n, d = x.shape
    out = []
    for c in scales:
        c = float(c)
        off = diag = 0.0
        for i in range(n):
            for j in range(n):
                dl = x[i] - x[j]
                r2 = float(dl @ dl)
                u = float(_u(kernel, c, d, r2, float(s[i] @ s[j]), float((s[i] - s[j]) @ dl) + d))
                if i == j:
                    diag += u
                else:
                    off += u
        out.append([off / (n * (n - 1)), (off + diag) / (n * n)])
    return np.array(out)


def gaussian_shift_ksd2(m, sigma):
    """Population KSD^2 of q = N(m, I_d) against p = N(0, I_d) for the Gaussian kernel of width sigma:
    |m|^2 (1 + 2 / sigma^2)^(-d / 2)."""
    m = np.asarray(m, dtype=np.float64)
    return float(m @ m) * (1.0 + 2.0 / sigma ** 2) ** (-len(m) / 2.0)
