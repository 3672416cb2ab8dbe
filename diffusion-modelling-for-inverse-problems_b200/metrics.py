"""Evaluation metrics computed next to the sampler (SURVEY.md §8f N2): the reference's 75-bin sample histograms and the
histogram KL it reports (`evaluate` in main_diffusion_linear.py:84-117 and main_diffusion_scatterometry.py:72-101),
on the GPU where the samples already are — `model(y, ..., return_tensor=True)` feeds them without a device->host copy.

    acc = HistogramKL(bins=(75, 75), ranges=((-3.5, 3.5), (-3.5, 3.5)))
    for repeat in range(10):
        acc.add(x_true, x_pred)          # CUDA tensors (n, d) — the reference's  hist_sum += np.histogramdd(...)
    kl2 = acc.kl()                       # sum(rel_entr(hist_true, hist_diffusion)) with the reference's normalisation

Beyond the reference: the unbiased Gaussian-kernel MMD^2 (Gretton et al. 2012), which needs no bins and works in any
dimension up to 16 —

    bw = median_bandwidth(x_true, x_pred)
    mmd = mmd2(x_true, x_pred, [bw / 2, bw, 2 * bw])      # float64 CUDA tensor (3,), one launch + one reduction

and the permutation two-sample test on it (the mixture kernel summed over the bandwidths), with a calibrated p-value —

    stat, p, null = mmd2_test(x_true, x_pred, [bw / 2, bw, 2 * bw], n_permutations=254)

and the kernel Stein discrepancy of samples against a target known through its score alone, which needs no
ground-truth samples (zero exactly when the samples come from the target) —

    ksd = ksd2(x_pred, score_posterior(x_pred, y), [0.5, 1.0, 2.0])      # float64 CUDA tensor (3,), IMQ kernel
"""
import math
import ctypes as C

import numpy as np
import torch

from . import _lib


MMD_MAX_DIM = 16
MMD_MAX_BW = 8
MMD_TEST_MAX_PERM = 254          # DMIP_MMD_TEST_MAX_PERM: permutations of one dmip_mmd_test call
MMD_TEST_MAX_POINTS = 1 << 20    # DMIP_MMD_TEST_MAX_POINTS: n + m


class DmipMmd(C.Structure):
    _fields_ = [("dim", C.c_int32), ("n_obs", C.c_int32), ("n", C.c_int64), ("m", C.c_int64), ("n_bw", C.c_int32),
                ("sigma", C.c_float * MMD_MAX_BW), ("x", C.c_void_p), ("y", C.c_void_p), ("out", C.c_void_p),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t)]


class DmipMmdTest(C.Structure):
    _fields_ = [("dim", C.c_int32), ("n_obs", C.c_int32), ("n", C.c_int64), ("m", C.c_int64), ("n_bw", C.c_int32),
                ("sigma", C.c_float * MMD_MAX_BW), ("n_perm", C.c_int32), ("x", C.c_void_p), ("y", C.c_void_p),
                ("labels", C.c_void_p), ("out", C.c_void_p), ("p_value", C.c_void_p), ("workspace", C.c_void_p),
                ("workspace_bytes", C.c_size_t)]


KSD_KERNELS = {"imq": 0, "gaussian": 1}   # DMIP_KSD_IMQ, DMIP_KSD_GAUSS


class DmipKsd(C.Structure):
    _fields_ = [("dim", C.c_int32), ("n_obs", C.c_int32), ("n", C.c_int64), ("kernel", C.c_int32),
                ("n_scales", C.c_int32), ("scale", C.c_float * MMD_MAX_BW), ("x", C.c_void_p), ("score", C.c_void_p),
                ("out", C.c_void_p), ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t)]


class DmipHistogram(C.Structure):
    _fields_ = [("dim", C.c_int32), ("bins", C.c_int32 * 4), ("edges", C.c_void_p * 4), ("n", C.c_int64),
                ("x", C.c_void_p), ("counts", C.c_void_p)]


def _bind():
    L = _lib.require_gpu()
    if not getattr(L, "_metrics_bound", False):
        L.dmip_histogramdd.restype = C.c_int
        L.dmip_histogramdd.argtypes = [C.POINTER(DmipHistogram), C.c_void_p]
        L.dmip_hist_kl.restype = C.c_int
        L.dmip_hist_kl.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_void_p, C.c_void_p]
        L.dmip_mmd_workspace_bytes.restype = C.c_size_t
        L.dmip_mmd_workspace_bytes.argtypes = [C.POINTER(DmipMmd)]
        L.dmip_mmd.restype = C.c_int
        L.dmip_mmd.argtypes = [C.POINTER(DmipMmd), C.c_void_p]
        L.dmip_mmd_test_workspace_bytes.restype = C.c_size_t
        L.dmip_mmd_test_workspace_bytes.argtypes = [C.POINTER(DmipMmdTest)]
        L.dmip_mmd_test.restype = C.c_int
        L.dmip_mmd_test.argtypes = [C.POINTER(DmipMmdTest), C.c_void_p]
        L.dmip_ksd_workspace_bytes.restype = C.c_size_t
        L.dmip_ksd_workspace_bytes.argtypes = [C.POINTER(DmipKsd)]
        L.dmip_ksd.restype = C.c_int
        L.dmip_ksd.argtypes = [C.POINTER(DmipKsd), C.c_void_p]
        L._metrics_bound = True
    return L


def histogramdd(x, bins, ranges, out=None):
    """np.histogramdd(x, bins=bins, range=ranges)[0] for a CUDA tensor x (n, d), bit-exact, as an int64 CUDA tensor of
    shape `bins`; with `out` the counts are accumulated into it."""
    L = _bind()
    if not x.is_cuda:
        raise RuntimeError("dmip metrics run on CUDA (sm_100a) only: there is no CPU fallback")
    x = x.detach().float().contiguous()
    n, dim = x.shape
    if len(bins) != dim or len(ranges) != dim:
        raise ValueError("The dimension of bins must be equal to the dimension of the sample x.")
    if out is None:
        out = torch.zeros(tuple(int(b) for b in bins), dtype=torch.int64, device=x.device)
    d = DmipHistogram()
    d.dim, d.n = dim, n
    keep = []
    for k in range(dim):
        e = torch.from_numpy(np.linspace(ranges[k][0], ranges[k][1], int(bins[k]) + 1)).to(x.device)   # float64, as numpy
        keep.append(e)
        d.bins[k] = int(bins[k])
        d.edges[k] = e.data_ptr()
    d.x, d.counts = x.data_ptr(), out.data_ptr()
    with torch.cuda.device(x.device):
        _lib.check(L.dmip_histogramdd(C.byref(d), _lib.stream_ptr()))
    return out


def hist_kl(hist_p, hist_q, epsilon=1e-10):
    """sum(scipy.special.rel_entr(p, q)) after the reference's normalisation (h / sum, + epsilon, / sum)."""
    L = _bind()
    assert hist_p.shape == hist_q.shape and hist_p.dtype == torch.int64 and hist_q.dtype == torch.int64
    out = torch.empty(3, dtype=torch.float64, device=hist_p.device)
    with torch.cuda.device(hist_p.device):
        _lib.check(L.dmip_hist_kl(hist_p.contiguous().data_ptr(), hist_q.contiguous().data_ptr(), hist_p.numel(),
                                  float(epsilon), out.data_ptr(), _lib.stream_ptr()))
    return out[0]


class HistogramKL:
    """Running pair of histograms over repeats and their KL — the inner loop of the reference's `evaluate`."""

    def __init__(self, bins, ranges, epsilon=1e-10):
        self.bins, self.ranges, self.epsilon = tuple(bins), tuple(ranges), epsilon
        self.hist_true = None
        self.hist_model = None

    def add(self, x_true, x_model):
        self.hist_true = histogramdd(x_true, self.bins, self.ranges, self.hist_true)
        self.hist_model = histogramdd(x_model, self.bins, self.ranges, self.hist_model)

    def kl(self, reverse=False):
        p, q = (self.hist_model, self.hist_true) if reverse else (self.hist_true, self.hist_model)
        return float(hist_kl(p, q, self.epsilon).item())


def _bandwidth_list(bandwidths, who="mmd2", what="bandwidths"):
    """1..MMD_MAX_BW positive finite kernel widths (`what` of `who`) as floats; raises ValueError otherwise."""
    try:
        bws = [float(b) for b in bandwidths]
    except TypeError:
        raise ValueError(f"{what} must be a sequence of numbers") from None
    if not 1 <= len(bws) <= MMD_MAX_BW:
        raise ValueError(f"{who} takes 1..{MMD_MAX_BW} {what}, got {len(bws)}")
    for b in bws:
        if not (math.isfinite(b) and b > 0):
            raise ValueError(f"{what} must be positive and finite, got {b!r}")
    return bws


def _sample_sets(x, y, who):
    """Shape checks shared by mmd2 and mmd2_test: (batched, n_obs, n, m, d); raises before any device work."""
    if not (torch.is_tensor(x) and torch.is_tensor(y)):
        raise ValueError("x and y must be tensors")
    if x.dim() != y.dim() or x.dim() not in (2, 3):
        raise ValueError(f"x and y must both be (n, d) or (n_obs, n, d), got shapes {tuple(x.shape)} and {tuple(y.shape)}")
    batched = x.dim() == 3
    xb, yb = (x, y) if batched else (x[None], y[None])
    n_obs, n, dim = xb.shape
    if yb.shape[0] != n_obs or yb.shape[2] != dim:
        raise ValueError(f"x {tuple(x.shape)} and y {tuple(y.shape)} differ in observations or dimension")
    m = yb.shape[1]
    if not 1 <= dim <= MMD_MAX_DIM:
        raise ValueError(f"{who} supports dimensions 1..{MMD_MAX_DIM}, got {dim}")
    if n < 2 or m < 2:
        raise ValueError(f"{who} needs at least 2 samples per set, got n = {n}, m = {m}")
    if n_obs < 1:
        raise ValueError(f"{who} needs at least one observation")
    return batched, n_obs, n, m, dim


def mmd2(x, y, bandwidths, *, terms=False):
    """Unbiased MMD^2 (Gretton et al. 2012, eq. 3) between the samples x and y for the Gaussian kernels
    k(a, b) = exp(-|a - b|^2 / (2 sigma^2)), one per entry of `bandwidths` (1..8 sigmas).

    x: (n, d) or (n_obs, n, d), y: (m, d) or (n_obs, m, d) CUDA tensors, d <= 16, n, m >= 2.  Returns a float64 CUDA tensor
    (..., n_bw) of MMD^2_u, or (..., n_bw, 4) holding {MMD^2_u, Kxx, Kyy, Kxy} with `terms=True`.  Kernel values are
    fp32, sums fp64; nothing synchronises with the host."""
    bws = _bandwidth_list(bandwidths)
    batched, n_obs, n, m, dim = _sample_sets(x, y, "mmd2")
    xb, yb = (x, y) if batched else (x[None], y[None])
    if not (x.is_cuda and y.is_cuda):
        raise RuntimeError("dmip metrics run on CUDA (sm_100a) only: there is no CPU fallback")
    L = _bind()
    xb = xb.detach().float().contiguous()
    yb = yb.detach().to(xb.device).float().contiguous()
    d = DmipMmd()
    d.dim, d.n_obs, d.n, d.m, d.n_bw = dim, n_obs, n, m, len(bws)
    for i, b in enumerate(bws):
        d.sigma[i] = b
    guard = _lib.Guarded()
    out = guard.empty(n_obs * len(bws) * 4, torch.float64, xb.device)
    ws_bytes = L.dmip_mmd_workspace_bytes(C.byref(d))
    ws = guard.empty(ws_bytes, torch.uint8, xb.device)
    d.x, d.y, d.out = xb.data_ptr(), yb.data_ptr(), out.data_ptr()
    d.workspace, d.workspace_bytes = ws.data_ptr(), ws_bytes
    with torch.cuda.device(xb.device):
        _lib.check(L.dmip_mmd(C.byref(d), _lib.stream_ptr()))
    guard.check("dmip_mmd")
    out = out.view(n_obs, len(bws), 4)
    if not terms:
        out = out[..., 0]
    return out if batched else out[0]


def permutation_labels(n_obs, n, m, n_permutations, *, generator=None, device="cuda"):
    """Random splits of n + m pooled points into n and m, packed as dmip_mmd_test takes them: an int32 tensor
    (n_obs, n_permutations, ceil((n + m) / 32)) whose bit j (word j // 32, bit j % 32) is set when pooled point j is in the
    first group.  Uniform random keys from `generator` on the device, argsort, the n smallest keys form the first group."""
    N = n + m
    W = -(-N // 32)
    out = torch.empty(n_obs, n_permutations, W, dtype=torch.int32, device=device)
    weights = torch.pow(2, torch.arange(32, device=device, dtype=torch.int64))
    rows = max(1, (1 << 25) // N)                       # bounds the key / index buffers to ~2^25 entries
    flat = out.view(-1, W)
    for r0 in range(0, flat.shape[0], rows):
        r1 = min(flat.shape[0], r0 + rows)
        keys = torch.rand(r1 - r0, N, device=device, generator=generator)
        first = torch.zeros(r1 - r0, W * 32, dtype=torch.int64, device=device)
        first.scatter_(1, keys.argsort(dim=1)[:, :n], 1)
        words = (first.view(r1 - r0, W, 32) * weights).sum(-1)
        flat[r0:r1] = torch.where(words >= 1 << 31, words - (1 << 32), words).to(torch.int32)
    return out


def mmd2_permutation_statistics(x, y, bandwidths, labels):
    """One dmip_mmd_test call: (out, p_value) float64 CUDA tensors of shapes (n_obs, P + 1) and (n_obs,) for the
    relabelings `labels` (n_obs, P, ceil((n + m) / 32)) int32 / uint32 bits, 1 <= P <= MMD_TEST_MAX_PERM.  out[:, 0] is
    MMD^2_u of x against y for the mixture kernel sum_b exp(-|a - c|^2 / (2 sigma_b^2)), out[:, 1 + p] that of
    permutation p; a label row without exactly n bits set gives NaN (and a NaN p-value).  x, y as for mmd2."""
    bws = _bandwidth_list(bandwidths, "mmd2_test")
    batched, n_obs, n, m, dim = _sample_sets(x, y, "mmd2_test")
    if n + m > MMD_TEST_MAX_POINTS:
        raise ValueError(f"mmd2_test takes at most {MMD_TEST_MAX_POINTS} pooled points, got n + m = {n + m}")
    W = -(-(n + m) // 32)
    if not torch.is_tensor(labels) or labels.dim() != 3 or labels.shape[0] != n_obs or labels.shape[2] != W:
        raise ValueError(f"labels must be ({n_obs}, n_permutations, {W}), got "
                         f"{tuple(labels.shape) if torch.is_tensor(labels) else type(labels).__name__}")
    if labels.dtype not in (torch.int32, torch.uint32):
        raise ValueError(f"labels must be int32 or uint32 bit words, got {labels.dtype}")
    P = labels.shape[1]
    if not 1 <= P <= MMD_TEST_MAX_PERM:
        raise ValueError(f"one call takes 1..{MMD_TEST_MAX_PERM} permutations, got {P}")
    if not (x.is_cuda and y.is_cuda and labels.is_cuda):
        raise RuntimeError("dmip metrics run on CUDA (sm_100a) only: there is no CPU fallback")
    L = _bind()
    xb, yb = (x, y) if batched else (x[None], y[None])
    xb = xb.detach().float().contiguous()
    yb = yb.detach().to(xb.device).float().contiguous()
    lab = labels.to(xb.device).contiguous()
    d = DmipMmdTest()
    d.dim, d.n_obs, d.n, d.m, d.n_bw, d.n_perm = dim, n_obs, n, m, len(bws), P
    for i, b in enumerate(bws):
        d.sigma[i] = b
    guard = _lib.Guarded()
    out = guard.empty(n_obs * (P + 1), torch.float64, xb.device)
    pv = guard.empty(n_obs, torch.float64, xb.device)
    ws_bytes = L.dmip_mmd_test_workspace_bytes(C.byref(d))
    ws = guard.empty(ws_bytes, torch.uint8, xb.device)
    d.x, d.y, d.labels, d.out, d.p_value = xb.data_ptr(), yb.data_ptr(), lab.data_ptr(), out.data_ptr(), pv.data_ptr()
    d.workspace, d.workspace_bytes = ws.data_ptr(), ws_bytes
    with torch.cuda.device(xb.device):
        _lib.check(L.dmip_mmd_test(C.byref(d), _lib.stream_ptr()))
    guard.check("dmip_mmd_test")
    return out.view(n_obs, P + 1), pv


def mmd2_test(x, y, bandwidths, n_permutations=254, *, generator=None):
    """Permutation two-sample test on MMD^2_u (Gretton et al. 2012, §5) with the mixture kernel
    sum_b exp(-|a - c|^2 / (2 sigma_b^2)) over `bandwidths` (1..8 sigmas) — the kernel whose value is
    mmd2(x, y, bandwidths).sum(-1).

    x: (n, d) or (n_obs, n, d), y: (m, d) or (n_obs, m, d) CUDA tensors as for mmd2, n + m <= 2^20.  Returns float64 CUDA
    tensors (stat, p_value, null) of shapes (...,), (...,) and (..., n_permutations): the observed statistic, the p-value
    (1 + #{null >= stat}) / (n_permutations + 1) and the statistics of the relabelings.  The permutations come from
    `generator` (a torch.Generator on the samples' device; None: the device's default generator).  Each call of the kernel
    takes up to 254 permutations; more run as several calls whose exceedance counts add."""
    bws = _bandwidth_list(bandwidths, "mmd2_test")
    batched, n_obs, n, m, dim = _sample_sets(x, y, "mmd2_test")
    if n + m > MMD_TEST_MAX_POINTS:
        raise ValueError(f"mmd2_test takes at most {MMD_TEST_MAX_POINTS} pooled points, got n + m = {n + m}")
    if isinstance(n_permutations, bool) or not isinstance(n_permutations, int) or n_permutations < 1:
        raise ValueError(f"n_permutations must be a positive integer, got {n_permutations!r}")
    if not (x.is_cuda and y.is_cuda):
        raise RuntimeError("dmip metrics run on CUDA (sm_100a) only: there is no CPU fallback")
    xb, yb = (x, y) if batched else (x[None], y[None])
    stat, nulls = None, []
    for p0 in range(0, n_permutations, MMD_TEST_MAX_PERM):
        P = min(MMD_TEST_MAX_PERM, n_permutations - p0)
        labels = permutation_labels(n_obs, n, m, P, generator=generator, device=xb.device)
        out, _ = mmd2_permutation_statistics(xb, yb, bws, labels)
        if stat is None:
            stat = out[:, 0]
        nulls.append(out[:, 1:])
    null = torch.cat(nulls, dim=1)
    exceed = (null >= stat[:, None]).sum(-1)
    p = (1.0 + exceed.double()) / (n_permutations + 1)
    p = torch.where(null.isnan().any(-1), torch.full_like(p, float("nan")), p)
    return (stat, p, null) if batched else (stat[0], p[0], null[0])


def ksd2(x, score, scales, kernel="imq", *, terms=False):
    """Kernel Stein discrepancy KSD^2 of the samples x against the target p whose score grad log p at x is `score`
    (Liu, Lee & Jordan 2016; Chwialkowski, Strathmann & Gretton 2016), one value per entry of `scales` (1..8):
    kernel='imq':      k = (c^2 + |a - b|^2)^(-1/2) with c = scale (detects non-convergence, Gorham & Mackey 2017);
    kernel='gaussian': k = exp(-|a - b|^2 / (2 sigma^2)) with sigma = scale.

    x, score: (n, d) or (n_obs, n, d) CUDA tensors of the same shape, d <= 16, n >= 2.  Returns a float64 CUDA tensor
    (..., n_scales) of the U-statistic KSD^2_U = mean_{i != j} u(x_i, x_j), or (..., n_scales, 2) holding
    {KSD^2_U, KSD^2_V} with `terms=True` (V: the mean over all pairs, i = j included; >= 0).  Pair values are fp32, sums
    fp64; a non-finite score gives NaN.  Nothing synchronises with the host."""
    cs = _bandwidth_list(scales, "ksd2", "scales")
    if kernel not in KSD_KERNELS:
        raise ValueError(f"ksd2 kernel must be one of {sorted(KSD_KERNELS)}, got {kernel!r}")
    if not (torch.is_tensor(x) and torch.is_tensor(score)):
        raise ValueError("x and score must be tensors")
    if x.shape != score.shape or x.dim() not in (2, 3):
        raise ValueError(f"x and score must have the same shape, (n, d) or (n_obs, n, d), got {tuple(x.shape)} and "
                         f"{tuple(score.shape)}")
    batched = x.dim() == 3
    xb, sb = (x, score) if batched else (x[None], score[None])
    n_obs, n, dim = xb.shape
    if not 1 <= dim <= MMD_MAX_DIM:
        raise ValueError(f"ksd2 supports dimensions 1..{MMD_MAX_DIM}, got {dim}")
    if n < 2:
        raise ValueError(f"ksd2 needs at least 2 samples per observation, got n = {n}")
    if n_obs < 1:
        raise ValueError("ksd2 needs at least one observation")
    if not (x.is_cuda and score.is_cuda):
        raise RuntimeError("dmip metrics run on CUDA (sm_100a) only: there is no CPU fallback")
    L = _bind()
    xb = xb.detach().float().contiguous()
    sb = sb.detach().to(xb.device).float().contiguous()
    d = DmipKsd()
    d.dim, d.n_obs, d.n, d.kernel, d.n_scales = dim, n_obs, n, KSD_KERNELS[kernel], len(cs)
    for i, c in enumerate(cs):
        d.scale[i] = c
    guard = _lib.Guarded()
    out = guard.empty(n_obs * len(cs) * 2, torch.float64, xb.device)
    ws_bytes = L.dmip_ksd_workspace_bytes(C.byref(d))
    ws = guard.empty(ws_bytes, torch.uint8, xb.device)
    d.x, d.score, d.out = xb.data_ptr(), sb.data_ptr(), out.data_ptr()
    d.workspace, d.workspace_bytes = ws.data_ptr(), ws_bytes
    with torch.cuda.device(xb.device):
        _lib.check(L.dmip_ksd(C.byref(d), _lib.stream_ptr()))
    guard.check("dmip_ksd")
    out = out.view(n_obs, len(cs), 2)
    if not terms:
        out = out[..., 0]
    return out if batched else out[0]


def median_bandwidth(x, y, max_points=4096):
    """The median heuristic: the median pairwise Euclidean distance (torch.median, i.e. the lower median) over at most
    `max_points` points taken with a fixed stride from the pooled samples of x and y ((..., d) tensors).  Plain torch on
    the tensors' device; returns a Python float."""
    d = x.shape[-1]
    pooled = torch.cat([x.detach().reshape(-1, d), y.detach().reshape(-1, d).to(x.device)]).double()
    stride = max(1, -(-pooled.shape[0] // int(max_points)))
    sub = pooled[::stride]
    dist = torch.cdist(sub, sub, compute_mode="donot_use_mm_for_euclid_dist")
    iu = torch.triu_indices(sub.shape[0], sub.shape[0], offset=1, device=sub.device)
    return float(dist[iu[0], iu[1]].median())
