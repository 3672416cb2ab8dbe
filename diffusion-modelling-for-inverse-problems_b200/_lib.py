"""ctypes binding of libdmip_sm100.so (C ABI: include/dmip.h).

PyTorch is plumbing here: it owns device memory and the CUDA stream; every kernel is ours.
There is no CPU or eager fallback: if the library is missing or the device is not sm_100, calls raise.
"""
import ctypes as C
import math
import os
import subprocess

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.environ.get("DMIP_LIB") or os.path.join(_HERE, "libdmip_sm100.so")   # DMIP_LIB: experiment builds
_lib = None

MAX_LAYERS = 8
PREC_F32, PREC_BF16 = 0, 1
CDE, CDIFFE, DPS = 0, 1, 2
RNG_PHILOX, RNG_INJECTED = 0, 1
SDE_VP, SDE_VE = 0, 1
_PREC = {"fp32": PREC_F32, "f32": PREC_F32, "float32": PREC_F32, "bf16": PREC_BF16, "bfloat16": PREC_BF16}


class DmipMlp(C.Structure):
    _fields_ = [("n_layers", C.c_int32), ("in_dim", C.c_int32), ("out_dim", C.c_int32),
                ("width", C.c_int32 * MAX_LAYERS),
                ("W", C.c_void_p * MAX_LAYERS), ("b", C.c_void_p * MAX_LAYERS)]


class DmipSampler(C.Structure):
    _fields_ = [("variant", C.c_int32), ("precision", C.c_int32), ("xdim", C.c_int32), ("ydim", C.c_int32),
                ("n_obs", C.c_int32), ("n_per_obs", C.c_int64), ("num_steps", C.c_int32),
                ("T", C.c_float), ("beta_min", C.c_float), ("beta_max", C.c_float),
                ("mean", C.c_float), ("std", C.c_float),
                ("net", DmipMlp), ("net2", DmipMlp),
                ("packed", C.c_void_p), ("packed2", C.c_void_p), ("l0_split", C.c_int32),
                ("y", C.c_void_p), ("out", C.c_void_p),
                ("rng_mode", C.c_int32), ("seed", C.c_uint64), ("gidx_base", C.c_uint64),
                ("x0", C.c_void_p), ("noise", C.c_void_p), ("ynoise", C.c_void_p),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
                ("sde_kind", C.c_int32), ("sigma_min", C.c_float), ("sigma_max", C.c_float),
                ("n_corrector", C.c_int32), ("snr", C.c_float)]


class DmipForward(C.Structure):
    _fields_ = [("precision", C.c_int32), ("net", DmipMlp), ("packed", C.c_void_p), ("l0_split", C.c_int32),
                ("n", C.c_int64), ("x_dim", C.c_int32), ("cond_dim", C.c_int32),
                ("x", C.c_void_p), ("cond", C.c_void_p), ("t", C.c_void_p), ("out", C.c_void_p),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t)]


def sde_params(base_sde):
    """(sde_kind, p0, p1) of a forward SDE as the kernels take it: (SDE_VP, beta_min, beta_max) or (SDE_VE, sigma_min,
    sigma_max).  The one place that decides which SDE a sampler or a fused loss runs."""
    from . import sdes
    if isinstance(base_sde, sdes.VarianceExplodingSDE):
        smin, smax = float(base_sde.sigma_min), float(base_sde.sigma_max)
        if not (math.isfinite(smin) and math.isfinite(smax) and 0.0 < smin < smax):
            raise ValueError(f"VE-SDE needs finite 0 < sigma_min < sigma_max (got sigma_min = {smin}, sigma_max = {smax})")
        return SDE_VE, smin, smax
    if hasattr(base_sde, 'beta_min') and hasattr(base_sde, 'beta_max'):     # VariancePreservingSDE and look-alikes
        return SDE_VP, float(base_sde.beta_min), float(base_sde.beta_max)
    raise ValueError("the kernels integrate the VP-SDE (beta_min, beta_max) or sdes.VarianceExplodingSDE, got "
                     f"{type(base_sde).__name__}")


def set_sde(desc, base_sde):
    """Fill the SDE fields (beta_min, beta_max, sde_kind, sigma_min, sigma_max) of a DmipSampler / DmipLoss /
    DmipPosteriorLoss descriptor from `base_sde`; the fields of the other SDE stay zero."""
    kind, p0, p1 = sde_params(base_sde)
    desc.sde_kind = kind
    if kind == SDE_VE:
        desc.sigma_min, desc.sigma_max = p0, p1
    else:
        desc.beta_min, desc.beta_max = p0, p1


def library_path():
    return _LIB_PATH


def build(verbose=False):
    """Compile libdmip_sm100.so in-tree with nvcc for sm_100a (works without a GPU)."""
    r = subprocess.run(["bash", os.path.join(_HERE, "csrc", "build.sh")], capture_output=True, text=True)
    if verbose or r.returncode:
        print(r.stdout, r.stderr)
    if r.returncode:
        raise RuntimeError("building libdmip_sm100.so failed:\n" + r.stdout + r.stderr)
    return _LIB_PATH


def lib():
    """Load the shared library (no compute).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise RuntimeError(f"{_LIB_PATH} is missing — run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(there is no CPU fallback)")
        L = C.CDLL(_LIB_PATH)
        L.dmip_version.restype = C.c_int
        L.dmip_last_error.restype = C.c_char_p
        L.dmip_device_ok.restype = C.c_int
        L.dmip_last_launch_count.restype = C.c_int
        L.dmip_pack_bytes.restype = C.c_size_t
        L.dmip_pack_bytes.argtypes = [C.POINTER(DmipMlp), C.c_int32, C.c_int32, C.c_int32]
        L.dmip_pack_mlp.restype = C.c_int
        L.dmip_pack_mlp.argtypes = [C.POINTER(DmipMlp), C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_size_t,
                                    C.c_void_p]
        L.dmip_sampler_workspace_bytes.restype = C.c_size_t
        L.dmip_sampler_workspace_bytes.argtypes = [C.POINTER(DmipSampler)]
        L.dmip_sampler_em_vp.restype = C.c_int
        L.dmip_sampler_em_vp.argtypes = [C.POINTER(DmipSampler), C.c_void_p]
        L.dmip_forward_workspace_bytes.restype = C.c_size_t
        L.dmip_forward_workspace_bytes.argtypes = [C.POINTER(DmipForward)]
        L.dmip_mlp_forward.restype = C.c_int
        L.dmip_mlp_forward.argtypes = [C.POINTER(DmipForward), C.c_void_p]
        _lib = L
    return _lib


def is_available():
    """True when the library is built, a CUDA device is visible and it is sm_100."""
    try:
        return torch.cuda.is_available() and bool(lib().dmip_device_ok())
    except Exception:
        return False


def check(rc):
    if rc != 0:
        msg = lib().dmip_last_error().decode()
        if rc == -1:
            raise ValueError(msg)
        raise RuntimeError(f"dmip error {rc}: {msg}")


def require_gpu():
    if not torch.cuda.is_available():
        raise RuntimeError("dmip needs a CUDA device (sm_100a): there is no CPU fallback")
    L = lib()
    if not L.dmip_device_ok():
        raise RuntimeError("dmip needs an sm_100 (B200) device: there is no fallback for other GPUs")
    return L


def precision_code(p):
    if isinstance(p, int):
        return p
    try:
        return _PREC[p.lower()]
    except KeyError:
        raise ValueError(f'No valid precision specified. Has to be one of "bf16" or "fp32", but {p!r} was given')


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def linear_layers(net):
    """The nn.Linear modules of an MLP in evaluation order (state_dict keys 0,3,5,7; SURVEY.md Q2)."""
    return [m for m in net.children() if isinstance(m, torch.nn.Linear)]


def mlp_desc(net, keep):
    """Fill a DmipMlp from an MLP/MLP2 module.  `keep` receives the tensors whose pointers are used."""
    layers = linear_layers(net)
    if len(layers) > MAX_LAYERS:         # the descriptor has MAX_LAYERS slots; fewer than 2 layers the library rejects itself
        raise ValueError(f"the library's kernels serve nets of at most {MAX_LAYERS} Linear layers (DMIP_MAX_LAYERS), "
                         f"got {len(layers)}")
    d = DmipMlp()
    d.n_layers = len(layers)
    d.in_dim = layers[0].in_features
    d.out_dim = layers[-1].out_features
    for i, lin in enumerate(layers):
        W = lin.weight.detach()
        b = lin.bias.detach()
        if not (W.is_cuda and W.dtype == torch.float32):
            raise RuntimeError("score-net parameters must be float32 CUDA tensors (no CPU fallback)")
        W = W.contiguous()
        b = b.contiguous()
        keep += [W, b]
        d.width[i] = lin.out_features
        d.W[i] = W.data_ptr()
        d.b[i] = b.data_ptr()
    return d


def mlp_desc_cached(net):
    """`mlp_desc` once per set of parameter storages: (descriptor, kept tensors).  Optimizer steps update the parameters in
    place, so during training the pointers — all the descriptor holds — do not change from step to step."""
    layers = linear_layers(net)
    key = tuple(p.data_ptr() for lin in layers for p in (lin.weight, lin.bias))
    hit = net.__dict__.get('_dmip_desc')
    if hit is None or hit[0] != key:
        keep = []
        hit = net.__dict__['_dmip_desc'] = (key, mlp_desc(net, keep), keep)
    return hit[1], hit[2]


class PackedNet:
    """Cache of the tcgen05 operand image of one net; re-packed when a parameter changes.

    "Changes" are detected through (data_ptr, tensor version): optimizer steps, `load_state_dict`, `copy_` and every
    other in-place op on the parameter bump the version.  Writes THROUGH `p.data` (EMA, manual clipping) do not — call
    `invalidate()` (or `model.invalidate_packed()`) after such an update."""

    def __init__(self):
        self.key = None
        self.buf = None

    def invalidate(self):
        """Force a re-pack at the next use."""
        self.key = None

    def get(self, net, n_varying, out_rows, split):
        L = require_gpu()
        layers = linear_layers(net)
        key = (n_varying, out_rows, split) + tuple((p.data_ptr(), p._version) for lin in layers
                                                   for p in (lin.weight, lin.bias))
        if key != self.key:
            keep = []
            d = mlp_desc(net, keep)
            nbytes = L.dmip_pack_bytes(C.byref(d), n_varying, out_rows, split)
            if nbytes == 0:
                check(-1)
            if self.buf is None or self.buf.numel() < nbytes:
                self.buf = torch.empty(nbytes, dtype=torch.uint8, device=layers[0].weight.device)
            check(L.dmip_pack_mlp(C.byref(d), n_varying, out_rows, split, C.c_void_p(self.buf.data_ptr()),
                                  nbytes, stream_ptr()))
            self.key = key
        return self.buf


class Guarded:
    """Debug allocator for kernel outputs and scratch (DMIP_GUARD=1): every buffer gets 4 KB of 0xA5 canary bytes in front
    and behind; `check()` synchronises and raises if a kernel wrote outside what it was given.  compute-sanitizer is
    closed on the GPU pool this was developed on (profiles/r02_compute_sanitizer_closed.txt) — this is the bounds check
    the test-suite runs instead (tests/gpu_cases.py case_guarded_buffers)."""
    PAD = 4096

    def __init__(self):
        self.on = os.environ.get("DMIP_GUARD", "") not in ("", "0")
        self.bufs = []

    def empty(self, n, dtype, device):
        if not self.on:
            return torch.empty(n, dtype=dtype, device=device)
        item = torch.empty(0, dtype=dtype).element_size()
        raw = torch.full((2 * self.PAD + n * item,), 0xA5, dtype=torch.uint8, device=device)
        self.bufs.append((raw, n * item))
        return raw[self.PAD:self.PAD + n * item].view(dtype)

    def check(self, what=""):
        if not self.on:
            return
        torch.cuda.synchronize()
        for raw, nbytes in self.bufs:
            ok = bool((raw[:self.PAD] == 0xA5).all()) and bool((raw[self.PAD + nbytes:] == 0xA5).all())
            if not ok:
                raise RuntimeError(f"dmip guard: a kernel wrote outside a {nbytes}-byte buffer ({what})")
        self.bufs = []


def tc_supported(net, n_varying=None, split=2):
    """True when the tcgen05 kernels can run this net: [in] -> 512 -> 512 -> 512 -> [out <= 128] and a layer-0 GEMM depth
    (the row-varying input columns, split `split` ways) of at most 512 — the conditions of tc_net_geom (csrc/dmip_pack.cu)."""
    layers = linear_layers(net)
    if not (len(layers) == 4 and all(l.out_features == 512 for l in layers[:3]) and layers[-1].out_features <= 128):
        return False
    dv = layers[0].in_features if n_varying is None else n_varying
    parts = 1 if split == 4 else split               # l0_split = 4: one f16 part
    k0 = (parts - 1) * ((dv + 7) // 8 * 8) + dv
    return (k0 + 15) // 16 * 16 <= 512
