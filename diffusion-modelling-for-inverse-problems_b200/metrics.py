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
"""
import math
import ctypes as C

import numpy as np
import torch

from . import _lib


MMD_MAX_DIM = 16
MMD_MAX_BW = 8


class DmipMmd(C.Structure):
    _fields_ = [("dim", C.c_int32), ("n_obs", C.c_int32), ("n", C.c_int64), ("m", C.c_int64), ("n_bw", C.c_int32),
                ("sigma", C.c_float * MMD_MAX_BW), ("x", C.c_void_p), ("y", C.c_void_p), ("out", C.c_void_p),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t)]


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


def _bandwidth_list(bandwidths):
    try:
        bws = [float(b) for b in bandwidths]
    except TypeError:
        raise ValueError("bandwidths must be a sequence of numbers") from None
    if not 1 <= len(bws) <= MMD_MAX_BW:
        raise ValueError(f"mmd2 takes 1..{MMD_MAX_BW} bandwidths, got {len(bws)}")
    for b in bws:
        if not (math.isfinite(b) and b > 0):
            raise ValueError(f"bandwidths must be positive and finite, got {b!r}")
    return bws


def mmd2(x, y, bandwidths, *, terms=False):
    """Unbiased MMD^2 (Gretton et al. 2012, eq. 3) between the samples x and y for the Gaussian kernels
    k(a, b) = exp(-|a - b|^2 / (2 sigma^2)), one per entry of `bandwidths` (1..8 sigmas).

    x: (n, d) or (n_obs, n, d), y: (m, d) or (n_obs, m, d) CUDA tensors, d <= 16, n, m >= 2.  Returns a float64 CUDA tensor
    (..., n_bw) of MMD^2_u, or (..., n_bw, 4) holding {MMD^2_u, Kxx, Kyy, Kxy} with `terms=True`.  Kernel values are
    fp32, sums fp64; nothing synchronises with the host."""
    bws = _bandwidth_list(bandwidths)
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
        raise ValueError(f"mmd2 supports dimensions 1..{MMD_MAX_DIM}, got {dim}")
    if n < 2 or m < 2:
        raise ValueError(f"mmd2 needs at least 2 samples per set, got n = {n}, m = {m}")
    if n_obs < 1:
        raise ValueError("mmd2 needs at least one observation")
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
