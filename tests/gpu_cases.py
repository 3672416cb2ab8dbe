"""GPU parity cases shared by the pytest suite (tests/test_gpu_*.py) and the staged diagnostic runner
(tests/gpu_diag.py).  Every case calls the CUDA path through the C ABI (ctypes) or through the drop-in classes and
compares with the CPU oracle / the reference-generated golden fixtures.  Tolerances are stated per case."""
import ctypes as C
import os
import numpy as np
import torch

import oracle
from oracle import nets as on, sampler as osamp
from oracle.weights import make_params, state_dict_from_params
from util import load_golden, meta_hidden

DEV = "cuda"


def _dmip():
    import dmip
    from dmip import _lib
    return dmip, _lib


# ------------------------------------------------------------------------------------------- tcgen05 building block
def case_umma(mode, n, k, seed=0):
    """128 x n x k bf16 GEMM via dmip_debug_umma (tools/probe).  bf16 products are exact in fp32, so only the summation order
    differs from the fp64 reference on bf16-rounded operands: tolerance 1e-4 * sqrt(k)."""
    _, _lib = _dmip()
    _lib.require_gpu()
    from tools.probe import probe     # building-block self-tests live outside the product library
    L = probe.lib()
    g = torch.Generator().manual_seed(seed)
    a = torch.randn(128, k, generator=g)
    w = torch.randn(n, k, generator=g)
    ref = (a.bfloat16().double() @ w.bfloat16().double().T).float()
    ad, wd = a.to(DEV), w.to(DEV)
    d = torch.full((128, n), float("nan"), device=DEV)
    probe.check(L.dmip_debug_umma(mode, ad.data_ptr(), wd.data_ptr(), d.data_ptr(), n, k, _lib.stream_ptr()))
    torch.cuda.synchronize()
    err = (d.cpu() - ref).abs().max().item()
    tol = 1e-4 * k ** 0.5
    return err, tol, dict(d=d.cpu(), ref=ref)


# ------------------------------------------------------------------------------------------- pack image
def sw128_offset(row, k, kblock_bytes=16384):
    kb, kin = k >> 6, k & 63
    chunk = (kin >> 3) ^ (row & 7)
    return kb * kblock_bytes + (row >> 3) * 1024 + (row & 7) * 128 + chunk * 16 + (kin & 7) * 2


def case_pack(xdim=3, ydim=23, out_dim=3, split=2, seed=3):
    """The packed image must hold exactly bf16(W) — f16(W0) for layer 0 with l0_split = 4 — at the swizzled positions the
    UMMA descriptor expects."""
    _, _lib = _dmip()
    L = _lib.require_gpu()
    in_dim = xdim + ydim + 1
    params = make_params(seed, in_dim, out_dim)
    from dmip.nets import MLP
    net = MLP(in_dim, out_dim, [512, 512, 512], torch.nn.Tanh())
    net.load_state_dict(state_dict_from_params(params))
    net.to(DEV)
    dv = xdim
    buf = _lib.PackedNet().get(net, dv, out_dim, split).cpu().numpy()
    dvp = (dv + 7) // 8 * 8
    parts = 1 if split == 4 else split              # l0_split = 4: one part, f16 instead of bf16
    k0 = (parts - 1) * dvp + dv
    k0pad = (k0 + 15) // 16 * 16
    kb0 = (k0pad + 63) // 64
    n_stages = 4 * kb0 + 72
    assert buf.size >= n_stages * 16384 + (1664 + 512 * (in_dim - dv)) * 4
    img = buf[: n_stages * 16384].view(np.uint16).reshape(n_stages, 8192)

    def bf16_bits(x):
        return (torch.as_tensor(x, dtype=torch.float32).bfloat16().view(torch.int16).numpy().astype(np.int64) & 0xFFFF)

    bad = 0
    W0, W1, W3 = params[0][0], params[1][0], params[3][0]
    hi = W0.bfloat16().float()
    lo = (W0 - hi).bfloat16().float()
    rng = np.random.default_rng(0)
    for _ in range(4000):
        r, k = int(rng.integers(128)), int(rng.integers(64))
        c, kb = int(rng.integers(4)), int(rng.integers(8))
        # layer 1, chunk c, K-block kb
        st = 4 * kb0 + c * 8 + kb
        got = int(img[st, sw128_offset(r, k) // 2])
        bad += got != int(bf16_bits(W1[c * 128 + r, kb * 64 + k]))
        # output layer
        st = 4 * kb0 + 64 + kb
        want = int(bf16_bits(W3[r, kb * 64 + k])) if r < out_dim else 0
        bad += int(img[st, sw128_offset(r, k) // 2]) != want
        # layer 0, chunk c, K-block 0
        st = c * kb0
        kg = k
        part, idx = divmod(kg, dvp)
        if part < parts and idx < dv:
            src = lo if part == 2 else hi
            if split == 4:
                want = int(W0[c * 128 + r, idx].half().view(torch.int16).item()) & 0xFFFF
            else:
                want = int(bf16_bits(src[c * 128 + r, idx]))
        else:
            want = 0
        bad += int(img[st, sw128_offset(r, k) // 2]) != want
    tail = buf[n_stages * 16384:].view(np.float32)
    ok_tail = np.array_equal(tail[:512], params[0][1].numpy()) and np.array_equal(tail[1536:1536 + out_dim], params[3][1].numpy()) \
        and np.array_equal(tail[1664:1664 + 512 * (in_dim - dv)].reshape(512, -1), W0[:, dv:].numpy())
    return bad + (0 if ok_tail else 1), 0, {}


# ------------------------------------------------------------------------------------------- score-net forward
def _load_net(cls_name, in_dim, out_dim, hidden, params):
    from dmip import nets
    net = getattr(nets, cls_name)(in_dim, out_dim, list(hidden), torch.nn.Tanh())
    net.load_state_dict(state_dict_from_params(params))
    return net.to(DEV)


def case_forward(name, precision):
    """a(x,y,t) vs the golden reference output.  fp32 path: 2e-5 (accumulation order).  bf16 path: operands rounded
    to bf16 (rel 2^-9) through 4 layers and tanh.approx (2^-11): tolerance 5e-3 * max|out|."""
    fx = load_golden(name)
    seed, xdim, ydim, out_dim = (int(v) for v in fx["meta"][:4])
    hidden = meta_hidden(fx, 4)
    params = make_params(seed, xdim + ydim + 1, out_dim, hidden)
    net = _load_net("MLP", xdim + ydim + 1, out_dim, hidden, params)
    net.precision = precision
    with torch.no_grad():
        out = net(fx["x"].to(DEV), fx["y"].to(DEV), fx["t"].to(DEV)).cpu()
    scale = fx["out"].abs().max().item()
    err = (out - fx["out"]).abs().max().item()
    tol = (2e-5 if precision == "fp32" else 5e-3) * scale
    return err, tol, dict(out=out, ref=fx["out"])


# ------------------------------------------------------------------------------------------- samplers
def _model(kind, xdim, ydim, hidden, seed):
    from dmip.models.diffusion import CDE, CDiffE, PosteriorDiffusionEstimator
    if kind == "CDE":
        m = CDE(xdim, ydim, list(hidden))
        m.sde.a.load_state_dict(state_dict_from_params(make_params(seed, xdim + ydim + 1, xdim, hidden)))
    elif kind == "CDiffE":
        m = CDiffE(xdim, ydim, list(hidden))
        m.sde.a.load_state_dict(state_dict_from_params(make_params(seed, xdim + ydim + 1, xdim + ydim, hidden)))
    else:
        m = PosteriorDiffusionEstimator(xdim, ydim, list(hidden))
        m.sde.a.prior_net.load_state_dict(state_dict_from_params(make_params(seed, xdim + 1, xdim, hidden)))
        m.sde.a.likelihood_net.load_state_dict(
            state_dict_from_params(make_params(seed + 100, xdim + ydim + 1, xdim, hidden)))
    m.sde.to(DEV)
    return m


def case_sampler(name, kind, precision, split=4):
    """Injected-noise sampler parity vs the golden reference samples.

    These fixtures use *untrained* nets, whose reverse dynamics expand (|x| reaches ~1e2) and amplify any
    perturbation, so the error is measured relative to max|x|: fp32 path 1e-5, bf16 path 2e-3
    (the contractive, trained case is `case_sampler_trained`)."""
    fx = load_golden(name)
    seed, xdim, ydim, N, S = (int(v) for v in fx["meta"][:5])
    m = _model(kind, xdim, ydim, meta_hidden(fx, 5), seed)
    m.l0_split = split
    mean, std = (fx["mean_std"].tolist() if "mean_std" in fx else (0.0, 1.0))
    inj = dict(x0=fx["x0"], noise=fx["noise"])
    if kind == "CDiffE":
        inj["ynoise"] = fx["ynoise"]
    out = torch.from_numpy(m(fx["y"], num_samples=N, num_steps=S, mean=mean, std=std, precision=precision, injected=inj))
    scale = fx["out"].abs().max().item()
    err = (out - fx["out"]).abs().max().item()
    tol = (1e-5 if precision == "fp32" else 2e-3) * scale
    return err, tol, dict(out=out, ref=fx["out"])


def trained_model():
    from dmip.models.diffusion import CDE
    fx = load_golden("trained_cde_linear")
    m = CDE(2, 2, [512, 512, 512])
    m.sde.a.load_state_dict({f"{k}.{n}": fx[f"{k}_{n}"] for k in (0, 3, 5, 7) for n in ("weight", "bias")})
    m.sde.to(DEV)
    return m


def case_sampler_trained(precision, mode):
    """Trained linear CDE, reference default S=200, N=512; noise = the keyed Philox stream.
    mode 'injected': the numpy-generated stream is fed in;  mode 'philox': the kernel generates it itself
    (gidx/step/quad keyed) — both must reproduce the reference samples.
    Tolerance: fp32 5e-4 (Philox transcendental intrinsics differ from numpy by ~1e-6 per draw, over 200 steps),
    bf16 1e-2 max abs (SURVEY.md §8d), plus mean shift <= 3e-3 and std ratio within 5e-3."""
    fx = load_golden("sampler_trained_cde_linear")
    N, S, seed = (int(v) for v in fx["philox"])
    m = trained_model()
    kw = {}
    if mode == "injected":
        gidx = np.arange(N)
        kw["injected"] = dict(
            x0=torch.from_numpy(oracle.philox.normals(gidx, oracle.philox.STEP_INIT, 0, 2, seed)),
            noise=torch.from_numpy(np.stack([oracle.philox.normals(gidx, i, 0, 2, seed) for i in range(S)])))
    else:
        kw["seed"] = seed
    out = torch.from_numpy(m(fx["y"], num_samples=N, num_steps=S, precision=precision, **kw))
    err = (out - fx["out"]).abs().max().item()
    tol = 5e-4 if precision == "fp32" else 1e-2
    dmean = (out.mean(0) - fx["out"].mean(0)).abs().max().item()
    rstd = (out.std(0) / fx["out"].std(0) - 1).abs().max().item()
    if precision == "bf16" and (dmean > 3e-3 or rstd > 5e-3):
        err = max(err, 1.0)
    return err, tol, dict(out=out, ref=fx["out"], dmean=dmean, rstd=rstd)


# ------------------------------------------------------------------------------------------- fused losses
LOSS_CASES = {
    # fixture: (model, kind, kwargs, weight gain)
    "loss_dsm_cde_linear": ("CDE", "DSM", {}, 1.0),
    "loss_dsm_cdiffe_linear": ("CDiffE", "DSM", {}, 1.0),
    "loss_dsm_cde_scat": ("CDE", "DSM", {}, 1.0),
    "loss_dsm_small": ("CDE", "DSM", {}, 1.0),
    "loss_pinn_cde_linear": ("CDE", "PINN", dict(lam=0.001, lam2=0.1, pde_loss="FPE", ic_metric="L2", pde_metric="L1"), 1.0),
    "loss_pinn_cde_linear_g3": ("CDE", "PINN", dict(lam=0.001, lam2=0.1, pde_loss="FPE", ic_metric="L2", pde_metric="L1"), 3.0),
    "loss_pinn_cde_linear_l2l1": ("CDE", "PINN", dict(lam=0.5, lam2=0.7, pde_loss="FPE", ic_metric="L1", pde_metric="L2"), 1.0),
    "loss_pinn_cde_linear_cfpe": ("CDE", "PINN", dict(lam=0.01, lam2=0.1, pde_loss="cScoreFPE", ic_metric="L2", pde_metric="L2"), 1.0),
    "loss_pinn_cde_scat": ("CDE", "PINN", dict(lam=0.01, lam2=0.001, pde_loss="FPE", ic_metric="L2", pde_metric="L1"), 1.0),
    "loss_pinn_cdiffe_linear": ("CDiffE", "PINN", dict(lam=0.001, lam2=0.1, pde_loss="FPE", ic_metric="L2", pde_metric="L1"), 1.0),
    "loss_pinn_small": ("CDE", "PINN", dict(lam=0.001, lam2=0.1, pde_loss="FPE", ic_metric="L2", pde_metric="L1"), 1.0),
    "loss_dsmpde_cde_linear": ("CDE", "DSM_PDE", dict(lam=0.1, pde_loss="FPE", pde_metric="L1"), 1.0),
    "loss_dsmpde_cde_linear_cfpe": ("CDE", "DSM_PDE", dict(lam=0.1, pde_loss="cScoreFPE", pde_metric="L1"), 1.0),
    # PINNLoss2 (losses.py:245-291) with the attribute its forward reads but never sets supplied (oracle/make_golden.py)
    "loss_pinn2_cde_linear": ("CDE", "PINN2", dict(lam=0.01, lam2=0.1, pde_loss="FPE", ic_metric="L2"), 1.0),
    "loss_pinn2_cde_scat_cfpe": ("CDE", "PINN2", dict(lam=0.02, lam2=0.05, pde_loss="cScoreFPE", ic_metric="L1"), 1.0),
    "loss_pinn_cdiffe_scat": ("CDiffE", "PINN", dict(lam=0.01, lam2=0.001, pde_loss="FPE", ic_metric="L2", pde_metric="L1"), 1.0),
    "loss_pinn_cde_scat_hutch": ("CDE", "PINN", dict(lam=0.01, lam2=0.001, pde_loss="FPE", ic_metric="L2", pde_metric="L1",
                                                     divergence_method="hutchinson"), 1.0),
    "loss_dsmpde_cdiffe_scat_hutch": ("CDiffE", "DSM_PDE", dict(lam=0.05, pde_loss="FPE", pde_metric="L2",
                                                                divergence_method="approx"), 1.0),
}


def case_loss(name, route=None):
    """Fused loss forward+backward (fp32 kernels) vs the reference's autograd result stored in the fixture:
    loss and every info-dict entry within 3e-4 relative; every parameter gradient within 3e-3 of its scale
    (atomics make the fp32 summation order of the batch reductions non-deterministic)."""
    from dmip import losses as dl
    from util import check_grads
    model_kind, kind, kw, gain = LOSS_CASES[name]
    if route is not None:       # 'exact_adjoint': the exact divergence through the grad_x reverse sweep instead of Q streams
        kw = dict(kw, divergence_method=route)
    fx = load_golden(name)
    seed, xdim, ydim, B = (int(v) for v in fx["meta"][:4])
    hidden = meta_hidden(fx, 4)
    from dmip.models.diffusion import CDE, CDiffE
    m = (CDE if model_kind == "CDE" else CDiffE)(xdim, ydim, list(hidden))
    out_dim = xdim if model_kind == "CDE" else xdim + ydim
    m.sde.a.load_state_dict(state_dict_from_params(make_params(seed, xdim + ydim + 1, out_dim, hidden, gain=gain)))
    m.sde.to(DEV)
    x, y, t, eps = (fx[k].to(DEV) for k in ("x", "y", "t", "eps"))
    info = {}
    if kind == "DSM":
        loss, _ = dl.dsm_fused(m, x, y, t, eps)
    else:
        if kind == "PINN":
            ic = fx["ic_target"].to(DEV)
            loss_fn = dl.PINNLoss(lambda xx, yy: ic, **kw)
        elif kind == "PINN2":
            ic = fx["ic_target"].to(DEV)
            loss_fn = dl.PINNLoss2(lambda xx, yy: ic, **kw)
        else:
            loss_fn = dl.DSM_PDELoss(**kw)
        if "probe" in fx:
            loss_fn.probe = fx["probe"].to(DEV)
        z = x if model_kind == "CDE" else torch.cat([x, y], 1)
        loss, info = loss_fn(m.sde, x, y, z, t, eps, None, None)
    m.sde.a.zero_grad()
    loss.backward()
    ref = fx["loss"].item()
    err = abs(loss.item() - ref) / max(abs(ref), 1e-6)
    for k, v in info.items():
        r = fx["info_" + k.replace(" ", "_").replace("-", "_")].item()
        err = max(err, abs(v.item() - r) / max(abs(r), 1e-6))
    lins = [mod for mod in m.sde.a.children() if isinstance(mod, torch.nn.Linear)]
    grads = [(l.weight.grad.cpu(), l.bias.grad.cpu()) for l in lins]
    try:
        check_grads(fx, grads, rtol=3e-3, atol_frac=3e-3)
    except AssertionError as e:
        print("  grad mismatch:", str(e)[:300])
        err = max(err, 1.0)
    return err, 3e-4, dict(loss=loss.item(), ref=ref)


def case_loss_path_taken():
    """kernel launches per fused PINN call on the linear CDE: tcgen05 path = pack + fwd + bwd + 4 wgrad = 7;
    FFMA path = 4 transposes + fwd + bwd + 4 wgrad (+ memset not counted) = 10."""
    import os
    from dmip import losses as dl
    from dmip.models.diffusion import CDE
    torch.manual_seed(0)
    m = CDE(2, 2, [512, 512, 512])
    m.sde.to(DEV)
    x, y, t = _dp_problem(512)
    counts = {}
    for path in ("tc", "ffma"):
        os.environ["DMIP_LOSS_PATH"] = path
        loss_fn = dl.PINNLoss(lambda xx, yy: -xx, lam=0.001, lam2=0.1, pde_loss="FPE", ic_metric="L2", pde_metric="L1")
        loss_fn(m.sde, x.to(DEV), y.to(DEV), x.to(DEV), t.to(DEV), torch.randn(512, 2, device=DEV), None, None)
        counts[path] = loss_fn.last_launch_count
    os.environ.pop("DMIP_LOSS_PATH", None)
    ok = counts["tc"] == 7 and counts["ffma"] == 10
    return (0.0 if ok else 1.0), 0.5, {k: float(v) for k, v in counts.items()}


# ------------------------------------------------------------------------------------------- scatterometry surrogate (K4)
def _surrogate_module():
    from util import surrogate_params
    sp = surrogate_params()
    fm = torch.nn.Sequential(torch.nn.Linear(3, 256), torch.nn.ReLU(), torch.nn.Linear(256, 256), torch.nn.ReLU(),
                             torch.nn.Linear(256, 256), torch.nn.ReLU(), torch.nn.Linear(256, 23))
    fm.load_state_dict({f"{i}.{n}": (W if n == "weight" else b) for i, (W, b) in zip((0, 2, 4, 6), sp)
                        for n in ("weight", "bias")})
    for p in fm.parameters():
        p.requires_grad = False
    return fm.to(DEV), sp


def _kink_rows(sp, x, thr=2e-5):
    """Rows with a hidden pre-activation (float64 oracle) within `thr` of the ReLU kink.  There the surrogate's Jacobian
    jumps by a finite amount, and which side a row falls on is decided by rounding: the reference's own fp32 autograd,
    the FFMA kernel and the bf16x3 tensor-core kernel (pre-activations to ~1e-5) may disagree — as two fp32 GEMM
    libraries would.  The gradient of such rows is not compared; the tests bound how many there are."""
    h = x.double()
    mn = torch.full((x.shape[0],), float("inf"), dtype=torch.float64)
    for W, b in sp[:-1]:
        z = h @ W.double().T + b.double()
        mn = torch.minimum(mn, z.abs().min(1).values)
        h = torch.relu(z)
    return mn < thr


def _surrogate_path(path):
    if path == "ffma":
        os.environ["DMIP_SURROGATE_PATH"] = "ffma"
    else:
        os.environ.pop("DMIP_SURROGATE_PATH", None)


def case_surrogate_energy(path="tc"):
    """get_log_posterior + energy_grad (utils_scatterometry.py:30-38, models/SNF.py:234-237) vs the reference's own
    autograd values in scat_energy.npz.  E rel 2e-4 (+1e-2: E ~ 1e3 from the 1/b^2 terms); grad 2e-4 of its scale;
    f(x): 1e-5 for the fp32 FFMA kernel (path 'ffma'), 2e-5 for the tensor-core kernel (bf16x3 split products: 16
    mantissa bits per operand, |f| <= 2), whose gradient is compared on the rows away from a ReLU kink (_kink_rows;
    at most 5 % of the fixture's rows are excluded)."""
    from dmip import utils_scatterometry as us
    fx = load_golden("scat_energy")
    fm, sp = _surrogate_module()
    _surrogate_path(path)
    try:
        E, g, f = us.surrogate_call(fm, fx["x"].to(DEV), fx["y"].to(DEV), 0.2, 0.01, 1000.0, want_fx=True)
        launches = us.surrogate_call.last_launch_count
        E, g, f = E.cpu(), g.cpu(), f.cpu()
        keep = torch.ones(fx["x"].shape[0], dtype=torch.bool) if path == "ffma" else ~_kink_rows(sp, fx["x"])
        e_k = 0.0 if keep.float().mean().item() >= 0.95 else 2.0
        e_f = (f - fx["fx"]).abs().max().item() / (1e-5 if path == "ffma" else 2e-5)
        e_E = ((E - fx["E"]).abs() / (2e-4 * fx["E"].abs() + 1e-2)).max().item()
        e_g = (g - fx["grad"])[keep].abs().max().item() / (2e-4 * fx["grad"].abs().max().item())
        # the tensor-core path is two launches (weight images, k_surrogate_tc), the FFMA path five (four transposes)
        e_l = 0.0 if launches == (2 if path == "tc" else 5) else 2.0
        # the public wrappers
        E2 = us.get_log_posterior(fx["x"].to(DEV), fm, 0.2, 0.01, fx["y"].to(DEV), 1000.0).cpu()
        s = us.make_score_posterior(fm, dict(a=0.2, b=0.01, lambd_bd=1000))(fx["x"].to(DEV), fx["y"].to(DEV)).cpu()
        e_w = max((E2 - E).abs().max().item(), (s + g).abs().max().item()) * 1e6
    finally:
        _surrogate_path("tc")
    return max(e_f, e_E, e_g, e_w, e_k, e_l), 1.0, dict(out=g, ref=fx["grad"], e_f=e_f, e_E=e_E, e_g=e_g, launches=launches)


def case_surrogate_vjp(path="tc"):
    """mode DMIP_SURR_LIK_VJP vs the oracle's explicit reverse sweep (oracle/scatterometry.py) — 2e-4 of the scale;
    also ragged row counts (n not a multiple of the 32-row / 128-row tile) and n = 1.  Tensor-core path: rows away from
    a ReLU kink (_kink_rows)."""
    from dmip import utils_scatterometry as us
    from oracle import scatterometry as oscat
    fx = load_golden("scat_energy")
    fm, sp = _surrogate_module()
    worst = 0.0
    _surrogate_path(path)
    try:
        for n in (512, 129, 77, 1):
            x, y = fx["x"][:n], fx["y"][:n]
            f = oscat.surrogate(sp, x)
            pre = (0.2 * f) ** 2 + 0.01 ** 2
            w = -0.04 * f / pre + (y - f) / pre + 0.04 * (y - f) ** 2 * f / pre
            ref = oscat.surrogate_vjp(sp, x, w)
            _, g, _ = us.surrogate_call(fm, x.to(DEV), y.to(DEV), 0.2, 0.01, mode=us.SURR_LIK_VJP)
            keep = torch.ones(n, dtype=torch.bool) if path == "ffma" else ~_kink_rows(sp, x)
            worst = max(worst, (g.cpu() - ref)[keep].abs().max().item() / (2e-4 * ref.abs().max().item()))
    finally:
        _surrogate_path("tc")
    return worst, 1.0, {}


def case_surrogate_observation_blocks(path="tc"):
    """rows_per_obs of the C ABI: y given as ONE row (the reference's broadcast of one observation over all samples,
    utils_scatterometry.py:30-38) or as 4 rows for 4 equal blocks of samples must give exactly what the expanded
    (n, ydim) tensor gives — same kernel, same arithmetic: bit-identical."""
    from dmip import utils_scatterometry as us
    fx = load_golden("scat_energy")
    fm, _ = _surrogate_module()
    x = fx["x"].to(DEV)
    worst = 0.0
    _surrogate_path(path)
    try:
        for k in (1, 4):
            yk = fx["y"][:k].to(DEV)
            full = yk.repeat_interleave(512 // k, dim=0)
            for mode in (us.SURR_ENERGY, us.SURR_LIK_VJP):
                a = us.surrogate_call(fm, x, yk, 0.2, 0.01, 1000.0, mode=mode, want_fx=True)
                b = us.surrogate_call(fm, x, full, 0.2, 0.01, 1000.0, mode=mode, want_fx=True)
                for u, v in zip(a, b):
                    if u is not None:
                        worst = max(worst, (u - v).abs().max().item())
        bad = 0.0
        try:
            us.surrogate_call(fm, x, fx["y"][:5].to(DEV), 0.2, 0.01, 1000.0)
            bad = 1.0            # 5 does not divide 512: must raise
        except ValueError:
            pass
    finally:
        _surrogate_path("tc")
    return max(worst, bad), 0.0, {}


def case_surrogate_other_shapes():
    """The tensor-core kernel's other admissible shapes — [in <= 3] -> 256 -> 256 -> 256 -> [out <= 32] — on random nets:
    (in 2, out 5), (in 1, out 16), (in 3, out 32), 1000 rows, against the FFMA kernel (same tolerances as above); and a
    net outside them ([3] -> 128 -> 128 -> [23]) must take the FFMA kernel (5 launches... here 4: three transposes)."""
    from dmip import utils_scatterometry as us
    worst, info = 0.0, {}
    for in_dim, out_dim in ((2, 5), (1, 16), (3, 32)):
        torch.manual_seed(10 * in_dim + out_dim)
        fm = torch.nn.Sequential(torch.nn.Linear(in_dim, 256), torch.nn.ReLU(), torch.nn.Linear(256, 256), torch.nn.ReLU(),
                                 torch.nn.Linear(256, 256), torch.nn.ReLU(), torch.nn.Linear(256, out_dim)).to(DEV)
        for p in fm.parameters():
            p.requires_grad = False
        sp = [(m.weight.detach().cpu(), m.bias.detach().cpu()) for m in fm if isinstance(m, torch.nn.Linear)]
        x = torch.rand(1000, in_dim) * 2.4 - 1.2
        with torch.no_grad():
            y = fm(x.to(DEV)) + 0.05 * torch.randn(1000, out_dim, device=DEV)
        keep = ~_kink_rows(sp, x)
        for mode in (us.SURR_ENERGY, us.SURR_LIK_VJP):
            _surrogate_path("tc")
            E, g, f = us.surrogate_call(fm, x.to(DEV), y, 0.2, 0.01, 1000.0, mode=mode, want_fx=True)
            n_tc = us.surrogate_call.last_launch_count
            _surrogate_path("ffma")
            try:
                E2, g2, f2 = us.surrogate_call(fm, x.to(DEV), y, 0.2, 0.01, 1000.0, mode=mode, want_fx=True)
            finally:
                _surrogate_path("tc")
            e_f = (f - f2).abs().max().item() / (1e-5 * max(1.0, f2.abs().max().item()))
            e_E = ((E - E2).abs() / (2e-4 * E2.abs() + 1e-2)).max().item() if E is not None else 0.0
            e_g = (g - g2).cpu()[keep].abs().max().item() / (2e-4 * g2.abs().max().item())
            info[f"{in_dim}_{out_dim}_{mode}"] = max(e_f, e_E, e_g)
            worst = max(worst, e_f, e_E, e_g, 0.0 if n_tc == 2 else 2.0, 0.0 if keep.float().mean().item() >= 0.9 else 2.0)
    small = torch.nn.Sequential(torch.nn.Linear(3, 128), torch.nn.ReLU(), torch.nn.Linear(128, 128), torch.nn.ReLU(),
                                torch.nn.Linear(128, 23)).to(DEV)
    us.surrogate_call(small, torch.rand(64, 3, device=DEV), torch.rand(64, 23, device=DEV), 0.2, 0.01, 1000.0)
    worst = max(worst, 0.0 if us.surrogate_call.last_launch_count == 4 else 2.0)
    return worst, 1.0, info


def case_surrogate_tc_vs_ffma(n=100003):
    """The tensor-core kernel against the fp32 FFMA kernel on `n` random rows of the prior box and beyond (|x| <= 1.2:
    boundary terms on), one observation per row — both modes, a ragged last tile, many tiles per CTA: f 2e-5, E 2e-4 rel
    (+1e-2), gradient 2e-4 of its scale on the rows away from a ReLU kink (at most 5 % excluded)."""
    from dmip import utils_scatterometry as us
    fx = load_golden("scat_energy")
    fm, sp = _surrogate_module()
    g = torch.Generator().manual_seed(1)
    x = torch.rand(n, 3, generator=g) * 2.4 - 1.2
    y = fx["y"][torch.randint(0, 512, (n,), generator=g)]
    keep = ~_kink_rows(sp, x)
    worst = 0.0 if keep.float().mean().item() >= 0.95 else 2.0
    info = {}
    for mode in (us.SURR_ENERGY, us.SURR_LIK_VJP):
        _surrogate_path("tc")
        E, gr, f = us.surrogate_call(fm, x.to(DEV), y.to(DEV), 0.2, 0.01, 1000.0, mode=mode, want_fx=True)
        _surrogate_path("ffma")
        try:
            E2, gr2, f2 = us.surrogate_call(fm, x.to(DEV), y.to(DEV), 0.2, 0.01, 1000.0, mode=mode, want_fx=True)
        finally:
            _surrogate_path("tc")
        e_f = (f - f2).abs().max().item() / 2e-5
        e_E = ((E - E2).abs() / (2e-4 * E2.abs() + 1e-2)).max().item() if E is not None else 0.0
        e_g = (gr - gr2).cpu()[keep].abs().max().item() / (2e-4 * gr2.abs().max().item())
        info[f"mode{mode}"] = (e_f, e_E, e_g)
        worst = max(worst, e_f, e_E, e_g)
    return worst, 1.0, info


def case_posterior_loss(name):
    """PosteriorLoss fused forward+backward vs the reference autograd values in the fixture: loss and both info
    entries 5e-4 relative, every parameter gradient of both nets within 3e-3 of its scale."""
    from dmip import losses as dl
    from dmip.models.diffusion import PosteriorDiffusionEstimator
    from util import check_grads
    fx = load_golden(name)
    seed, xdim, ydim, B = (int(v) for v in fx["meta"][:4])
    hid = meta_hidden(fx, 4)
    m = PosteriorDiffusionEstimator(xdim, ydim, list(hid))
    m.sde.a.prior_net.load_state_dict(state_dict_from_params(make_params(seed, xdim + 1, xdim, hid)))
    m.sde.a.likelihood_net.load_state_dict(state_dict_from_params(make_params(seed + 100, xdim + ydim + 1, xdim, hid)))
    m.sde.to(DEV)
    fm, _ = _surrogate_module()
    loss_fn = dl.PosteriorLoss(fm, 0.2, 0.01, float(fx["lam"]))
    loss, info = loss_fn(m.sde, fx["x"].to(DEV), fx["y"].to(DEV), fx["t"].to(DEV), fx["eps"].to(DEV))
    m.sde.a.zero_grad()
    loss.backward()
    ref = fx["loss"].item()
    err = abs(loss.item() - ref) / abs(ref)
    for k in ("PriorLoss", "LikelihoodLoss"):
        r = fx["info_" + k].item()
        err = max(err, abs(info[k].item() - r) / abs(r))
    for prefix, net in (("prior_", m.sde.a.prior_net), ("lik_", m.sde.a.likelihood_net)):
        lins = [mod for mod in net.children() if isinstance(mod, torch.nn.Linear)]
        grads = [(l.weight.grad.cpu(), l.bias.grad.cpu()) for l in lins]
        try:
            check_grads(fx, grads, prefix=prefix, rtol=3e-3, atol_frac=3e-3)
        except AssertionError as e:
            print("  grad mismatch:", prefix, str(e)[:300])
            err = max(err, 1.0)
    return err, 5e-4, dict(loss=loss.item(), ref=ref)


# ------------------------------------------------------------------------------------------- sharding / statistics
def case_shards_are_bit_identical(precision="bf16"):
    """Philox counters are keyed by the GLOBAL particle index: integrating [0,N) in one call or as three ragged shards
    with gidx_base = shard start gives bit-identical samples (what makes multi-GPU runs independent of the GPU count)."""
    m = trained_model()
    fx = load_golden("sampler_trained_cde_linear")
    N, S, seed = 1000, 40, 99
    full = m(fx["y"], num_samples=N, num_steps=S, precision=precision, seed=seed, return_tensor=True)
    parts, start = [], 0
    for count in (300, 129, 571):
        parts.append(m(fx["y"], num_samples=count, num_steps=S, precision=precision, seed=seed, gidx_base=start,
                       return_tensor=True))
        start += count
    err = (torch.cat(parts) - full).abs().max().item()
    # the same through the public sharding helper (world size 1 -> the whole range)
    from dmip.distributed import sample_sharded
    one = sample_sharded(m, fx["y"], num_samples=N, num_steps=S, seed=seed, precision=precision)
    err = max(err, (one - full).abs().max().item())
    return err, 0.0, {}


def case_batched_observations():
    """y of shape (n_obs, ydim): all observations in one launch == one call per observation with the matching
    global-index offset (config 4 layout: observation o occupies rows [o N, (o+1) N))."""
    m = trained_model()
    g = torch.Generator().manual_seed(5)
    ys = torch.randn(3, 2, generator=g)
    N, S, seed = 200, 30, 7
    batched = m(ys, num_samples=N, num_steps=S, seed=seed, return_tensor=True)
    assert batched.shape == (3, N, 2)
    err = 0.0
    for o in range(3):
        single = m(ys[o], num_samples=N, num_steps=S, seed=seed, gidx_base=o * N, return_tensor=True)
        err = max(err, (single - batched[o]).abs().max().item())
    return err, 0.0, {}


def case_posterior_statistics():
    """Statistics of the bf16 tensor-core sampler on the DSM-trained linear CDE, 65,536 particles, reference-default
    200 steps, in-kernel Philox noise, against (a) the fp32 kernel on the same noise and (b) the analytic posterior
    (linear_problem.py:41-46).  Tolerances: |mean shift| <= 3e-3 and |std ratio - 1| <= 5e-3 vs fp32 (SURVEY.md §8d);
    the reference's own quality metric — histogram KL with 75 bins on [-3.5, 3.5]^2 (main_diffusion_linear.py:86-117) —
    between the two precisions <= 2e-3 (two independent fp32 runs of this size differ by ~3e-2: sampling noise);
    mean / covariance vs the analytic posterior within the trained model's own error (0.08 / 0.05); and, on independent
    noise streams, KL(fp32 || bf16) <= 1.5 x KL(fp32 || fp32') at 131,072 particles (the SURVEY's statistical bar)."""
    import numpy as np
    fx = load_golden("sampler_trained_cde_linear")
    m = trained_model()
    N, S, seed = 65536, 200, 2024
    lo = m(fx["y"], num_samples=N, num_steps=S, precision="bf16", seed=seed)
    hi = m(fx["y"], num_samples=N, num_steps=S, precision="fp32", seed=seed)
    dmean = float(np.abs(lo.mean(0) - hi.mean(0)).max())
    rstd = float(np.abs(lo.std(0) / hi.std(0) - 1).max())

    def hist(a):
        h, _ = np.histogramdd(a, bins=(75, 75), range=((-3.5, 3.5), (-3.5, 3.5)))
        h = h / h.sum() + 1e-10
        return h / h.sum()

    p, q = hist(hi), hist(lo)
    kl = float((p * np.log(p / q)).sum())
    post_mean, post_cov = fx["post_mean"].numpy(), fx["post_cov"].numpy()
    emean = float(np.abs(lo.mean(0) - post_mean).max())
    ecov = float(np.abs(np.cov(lo.T) - post_cov).max())
    # SURVEY.md §8d, statistical tolerance: on INDEPENDENT noise streams the histogram KL between the new path and the
    # fp32 path must not exceed 1.5 x the KL between two independent fp32 runs (GPU-side histograms, dmip.metrics)
    from dmip import metrics as dmet
    bins, rng = (75, 75), ((-3.5, 3.5), (-3.5, 3.5))
    N2 = 131072
    sets = [m(fx["y"], num_samples=N2, num_steps=S, precision=prec, seed=sd, return_tensor=True)
            for prec, sd in (("bf16", 31), ("fp32", 32), ("fp32", 33))]
    h_new, h_ref, h_ref2 = (dmet.histogramdd(x, bins, rng) for x in sets)
    kl_new = float(dmet.hist_kl(h_ref, h_new))
    kl_ref = float(dmet.hist_kl(h_ref, h_ref2))
    err = max(dmean / 3e-3, rstd / 5e-3, kl / 2e-3, emean / 0.08, ecov / 0.05, kl_new / (1.5 * kl_ref))
    return err, 1.0, dict(dmean=dmean, rstd=rstd, kl=kl, emean=emean, ecov=ecov, kl_new=kl_new, kl_ref=kl_ref)


def case_edge_shapes():
    """Ragged and degenerate shapes through the public call: empty result, a single particle, one SDE step, particle
    counts that straddle the 128-row tile, a lone tile (the second CTA of the cluster runs masked), and an invalid
    argument.  bf16 path vs fp32 path on the same Philox stream, relative to max|x|: 2e-2 — with 1-3 SDE steps the step size
    delta*beta reaches 20 and amplifies the bf16 rounding of the net output (measured 1e-2 at S=3, 6e-4 at S=50): these
    cases check shapes and masking, the accuracy cases are `case_sampler_trained` / `case_posterior_statistics`."""
    import numpy as np
    m = trained_model()
    fx = load_golden("sampler_trained_cde_linear")
    y = fx["y"]
    out = m(y, num_samples=0, num_steps=5, seed=1)
    assert out.shape == (0, 2) and out.dtype == np.float32
    worst = 0.0
    for N, S in ((1, 1), (1, 7), (127, 3), (128, 3), (129, 3), (257, 2), (148 * 128 + 5, 2)):
        lo = m(y, num_samples=N, num_steps=S, precision="bf16", seed=3)
        hi = m(y, num_samples=N, num_steps=S, precision="fp32", seed=3)
        assert lo.shape == (N, 2) and np.isfinite(lo).all()
        worst = max(worst, float(np.abs(lo - hi).max() / np.abs(hi).max()))
    try:
        m(y, num_samples=4, num_steps=0, seed=1)
        worst = 1.0                                   # num_steps = 0 must be rejected (DMIP_EINVAL -> ValueError)
    except ValueError:
        pass
    return worst, 2e-2, {}


# ------------------------------------------------------------------------------------------- training loop (a10)
def case_train_epoch(loss_name, graph=False, capturable=False):
    """CDE.train_epoch with the reference's call signature (models/diffusion.py:74-105) on the linear toy problem
    (linear_problem.py:10-16: y = A x + b + 0.3 eps): Adam steps through the fused loss kernels must reduce the loss,
    and the DSM-trained net's posterior mean must move to the analytic posterior (linear_problem.py:41-46)."""
    import numpy as np
    from dmip import losses as dl
    from dmip.models.diffusion import CDE
    torch.manual_seed(0)
    A = torch.tensor([[1.0, 0.5], [-0.3, 1.2]])
    b = torch.tensor([0.2, -0.1])
    sig = 0.3
    g = torch.Generator().manual_seed(7)
    X = torch.randn(16000, 2, generator=g)
    Y = X @ A.T + b + sig * torch.randn(16000, 2, generator=g)
    X, Y = X.to(DEV), Y.to(DEV)
    m = CDE(2, 2, [512, 512, 512])
    opt = torch.optim.Adam(m.sde.a.parameters(), lr=1e-3 if loss_name == "DSM" else 3e-4, capturable=capturable)
    if loss_name == "DSM":
        loss_fn = dl.DSMLoss()
    else:
        cov = torch.linalg.inv(torch.eye(2) + A.T @ A / sig ** 2).to(DEV)
        At_d, b_d, prec_t = A.T.to(DEV), b.to(DEV), torch.linalg.inv(cov).T.contiguous()

        def score_posterior(x, y):              # analytic posterior score (linear_problem.py:61-65), device code only
            mean = (cov @ (At_d @ (y - b_d).T / sig ** 2)).T
            return -(x - mean) @ prec_t

        loss_fn = dl.PINNLoss(score_posterior, lam=0.001, lam2=0.1, pde_loss="FPE", ic_metric="L2", pde_metric="L1")

    def loader():
        perm = torch.randperm(X.shape[0], device=DEV)
        for i in range(0, X.shape[0], 1000):
            idx = perm[i:i + 1000]
            yield X[idx], Y[idx]

    losses = []
    for epoch in range(12 if loss_name == "DSM" else 4):
        loss, info = m.train_epoch(opt, loss_fn, loader, graph=graph) if graph else m.train_epoch(opt, loss_fn, loader)
        losses.append(float(loss))
    assert all(np.isfinite(losses)), losses
    if graph:
        gs = m._graphed_step
        assert gs.step_in_graph == capturable and isinstance(gs.graph, torch.cuda.CUDAGraph)
    if loss_name != "DSM":
        assert set(info) == {"PDE-Loss", "Initial Condition", "DSM-Loss"}
        return (0.0 if losses[-1] < losses[0] else 1.0), 0.5, dict(first=losses[0], last=losses[-1])
    # posterior check for one observation
    y0 = torch.tensor([0.7, -0.4])
    cov = torch.linalg.inv(torch.eye(2) + A.T @ A / sig ** 2)
    mean = cov @ (A.T @ (y0 - b) / sig ** 2)
    xs = m(y0, num_samples=20000, num_steps=200, seed=11)
    emean = float(np.abs(xs.mean(0) - mean.numpy()).max())
    ok = losses[-1] < 0.8 * losses[0] and emean < 0.15
    return (0.0 if ok else 1.0), 0.5, dict(first=losses[0], last=losses[-1], emean=emean)


# ------------------------------------------------------------------------------------------- evaluation metrics (N2)
def case_histogram_kl():
    """GPU histogramdd / KL vs numpy + scipy (the reference's evaluate loop): counts bit-exact — including samples on
    bin edges, on the right-most edge, outside the range and NaN — for 2-D (linear, 75 bins on [-3.5, 3.5]) and 3-D
    (scatterometry, 75 bins on [-1.2, 1.2]); KL within 1e-12."""
    import numpy as np
    from dmip import metrics as dmet
    from oracle import metrics as omet
    rng = np.random.default_rng(0)
    worst = 0.0
    for dim, lim in ((2, 3.5), (3, 1.2)):
        bins, ranges = (75,) * dim, ((-lim, lim),) * dim
        edges = np.linspace(-lim, lim, 76)
        sets_true, sets_model = [], []
        acc = dmet.HistogramKL(bins, ranges)
        for rep in range(3):
            a = (rng.standard_normal((30000, dim)) * lim * 0.45).astype(np.float32)
            b = (rng.standard_normal((30000, dim)) * lim * 0.5 + 0.1).astype(np.float32)
            a[:200, 0] = edges[rng.integers(0, 76, 200)].astype(np.float32)      # exactly on edges (after fp32 rounding)
            a[200:210, 1] = np.float32(lim)                                      # right-most edge: inclusive
            a[210:215, 0] = np.float32(-lim)
            a[215:220, 1] = np.nan
            b[:50] *= 10.0                                                       # outliers
            sets_true.append(a)
            sets_model.append(b)
            acc.add(torch.from_numpy(a).to(DEV), torch.from_numpy(b).to(DEV))
        ht, hm = omet.hist_sum(sets_true, bins, ranges), omet.hist_sum(sets_model, bins, ranges)
        if not (np.array_equal(acc.hist_true.cpu().numpy(), ht.astype(np.int64))
                and np.array_equal(acc.hist_model.cpu().numpy(), hm.astype(np.int64))):
            return 1.0, 0.0, {}
        for rev in (False, True):
            ref = omet.kl2(hm, ht) if rev else omet.kl2(ht, hm)
            worst = max(worst, abs(acc.kl(reverse=rev) - ref))
    return worst, 1e-12, {}


# ------------------------------------------------------------------------------------------- Metropolis chains (N3)
def _chains_match(x, ref, de, de_ref):
    """fraction of chains that differ from the reference (an accept decision on a near-tie may flip in fp32) and the
    energy-difference error of the matching ones"""
    same = (x - ref).abs().max(1).values <= 2e-5
    bad_de = ((de[same] - de_ref[same]).abs() > 1e-3 * de_ref[same].abs() + 5e-2).float().mean().item()
    return 1.0 - same.float().mean().item() + bad_de


def case_metropolis(mode):
    """dmip.mcmc.anneal_to_energy vs the reference's anneal_to_energy (models/SNF.py:250-275) on the stored random
    stream (fixture mcmc_scat, 2 observations x 128 chains x 40 steps): >= 98 % of the chains end on the same point to
    2e-5 with the same energy difference.  mode 'philox': the in-kernel Philox stream must reproduce, bit for bit, the
    run fed with the numpy mirror of that stream."""
    from dmip import mcmc
    fm, _ = _surrogate_module()
    fx = load_golden("mcmc_scat")
    n_obs, n_per, S = (int(v) for v in fx["meta"])
    x0, ys = fx["x0"].to(DEV), fx["y"].to(DEV)
    std = float(fx["noise_std"])
    if mode == "injected":
        x, de = mcmc.anneal_to_energy(x0, fm, 0.2, 0.01, ys, 1000, S, std, injected=dict(noise=fx["noise"], unif=fx["unif"]))
        return _chains_match(x.cpu(), fx["out"], de.cpu(), fx["de"]), 0.02, {}
    seed, base = 4321, 1000
    gidx = np.arange(n_obs * n_per) + base
    noise = torch.from_numpy(np.stack([oracle.philox.normals(gidx, i, 2, 3, seed) for i in range(S)]))
    unif = torch.from_numpy(np.stack([oracle.philox.uniforms(gidx, i, 3, seed) for i in range(S)]))
    xa, dea = mcmc.anneal_to_energy(x0, fm, 0.2, 0.01, ys, 1000, S, std, seed=seed, gidx_base=base)
    xb, deb = mcmc.anneal_to_energy(x0, fm, 0.2, 0.01, ys, 1000, S, std, injected=dict(noise=noise, unif=unif))
    moved = ((xa - x0).abs().max(1).values > 0).float().mean().item()
    err = _chains_match(xa.cpu(), xb.cpu(), dea.cpu(), deb.cpu()) + (0.0 if moved > 0.5 else 1.0)
    return err, 0.02, dict(moved=moved)


def case_evaluate():
    """dmip.evaluation on the trained linear CDE: all observations in one sampler launch per repeat, histograms / KL /
    NLL / score MSE on the GPU.  The KL column must equal scipy's on the same accumulated counts (checked inside
    case_histogram_kl); here: the trained model is close to the analytic posterior (KL2 < 0.5 with 2 x 5000 samples in
    75 x 75 bins, |NLL gap| < 0.1) and the scatterometry variant runs end to end on generated ground truth."""
    from dmip import evaluation, mcmc
    from dmip.linear_problem import LinearForwardProblem
    from dmip.models.diffusion import CDE
    from dmip.utils_scatterometry import make_score_posterior
    m = trained_model()
    lin = LinearForwardProblem()
    g = torch.Generator().manual_seed(3)
    xs = torch.randn(6, 2, generator=g)
    ys = lin(xs) + 0.3 ** 0.5 * torch.randn(6, 2, generator=g)
    kl, nlpd, mse, table = evaluation.evaluate_linear(m, ys, lin, n_samples_x=5000, n_repeats=2)
    ok = kl < 0.5 and nlpd < 0.1 and np.isfinite(mse) and table['KL2'].shape == (6,)
    fm, _ = _surrogate_module()
    params = {'a': 0.2, 'b': 0.01, 'lambd_bd': 1000, 'xdim': 3, 'ydim': 23}
    xt = torch.rand(3, 3, generator=g) * 1.6 - 0.8
    with torch.no_grad():
        ysc = fm(xt.to(DEV))
    gt = mcmc.generate_gt_samples(fm, params, ysc, 2048, 60, 0.02, n_repeats=2, seed=11)
    torch.manual_seed(0)
    ms = CDE(3, 23, [512, 512, 512])
    ms.sde.to(DEV)
    # a short DSM fit so that the reverse SDE contracts (an untrained net sends every sample out of the histogram range
    # and the KL is 0/0, upstream too)
    from dmip import losses as dl
    X = torch.rand(8000, 3, device=DEV) * 2 - 1
    with torch.no_grad():
        fX = fm(X)
        Y = fX + 0.01 * torch.randn_like(fX) + 0.2 * fX * torch.randn_like(fX)
    opt = torch.optim.Adam(ms.sde.a.parameters(), lr=1e-3)
    for _ in range(25):
        ms.train_epoch(opt, dl.DSMLoss(), lambda: ((X[i:i + 1000], Y[i:i + 1000]) for i in range(0, 8000, 1000)))
    kl2, nlpd2, mse2, table2 = evaluation.evaluate_scatterometry(
        ms, ysc, fm, lambda i, j: gt[i, j], 2048, make_score_posterior(fm, params), 0.2, 0.01, 1000, n_repeats=2,
        num_steps=20)
    ok = ok and all(np.isfinite(v).all() for v in table2.values()) and set(table2) == {
        'KL2', 'KL_reverse', 'NLL_mcmc', 'NLL_diffusion', 'MSE'}
    return (0.0 if ok else 1.0), 0.5, dict(kl=float(kl), nlpd=float(nlpd), mse=float(mse), kl_scat=float(kl2))


def case_host_results_do_not_alias():
    """model(y) returns numpy arrays that live in pooled pinned buffers: an array the caller still holds must never be
    overwritten by a later call; a dropped one is recycled (no new pinned allocation)."""
    m = trained_model()
    y = torch.tensor([0.4, -0.7])
    x1 = m(y, num_samples=4096, num_steps=10, seed=1)
    keep = x1.copy()
    x2 = m(y, num_samples=4096, num_steps=10, seed=2)
    row = x2[5]                                   # a derived view keeps its parent buffer busy
    ok = np.array_equal(x1, keep) and not np.array_equal(x1, x2) and len(m._stage['pool']) == 2
    del x2
    x3 = m(y, num_samples=4096, num_steps=10, seed=3)
    ok = ok and len(m._stage['pool']) == 3 and np.array_equal(x1, keep)
    del x3, row
    x4 = m(y, num_samples=4096, num_steps=10, seed=1)
    ok = ok and len(m._stage['pool']) == 3 and np.array_equal(x4, keep) and np.array_equal(x1, keep)
    return (0.0 if ok else 1.0), 0.5, {}


# ------------------------------------------------------------------------------------------- data-parallel training (e2)
def _dp_problem(B=4096, seed=5):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, 2, generator=g)
    A = torch.tensor([[1.0, 0.5], [0.0, 1.0]])
    y = x @ A.T + torch.tensor([0.3, 0.5]) + 0.3 ** 0.5 * torch.randn(B, 2, generator=g)
    t = torch.rand(B, 1, generator=g) * 0.98 + 0.01
    return x, y, t


def _dp_model_and_loss(kind):
    from dmip import losses as dl
    from dmip.models.diffusion import CDE
    torch.manual_seed(0)
    m = CDE(2, 2, [512, 512, 512])
    if kind == "DSM":
        loss_fn = dl.DSMLoss()
    else:
        loss_fn = dl.PINNLoss(lambda xx, yy: -xx, lam=0.001, lam2=0.1, pde_loss="FPE", ic_metric="L2", pde_metric="L1")
    return m, loss_fn


def _dp_single_process_reference(kind, x, y, t, eps_seed):
    """loss and flat gradient of ONE process on the whole batch (the autograd route of train_epoch)"""
    from dmip.losses import fused_train_step
    m, loss_fn = _dp_model_and_loss(kind)
    torch.manual_seed(eps_seed)
    loss, info = fused_train_step(m, loss_fn, x.to(DEV), y.to(DEV), t.to(DEV))
    m.sde.a.zero_grad()
    loss.backward()
    flat = torch.cat([p.grad.reshape(-1) for p in m.sde.a.parameters()])
    return loss.detach(), flat


def case_data_parallel_emulated(kind):
    """Two data-parallel ranks emulated on ONE GPU: each shard is evaluated with batch_global = B into its own flat
    gradient bucket, the buckets are summed (what the all-reduce does) and compared with the single-process step on the
    concatenated batch: gradients within 2e-5 of their scale (+ the reduction-order noise of fp32 atomics), loss 1e-5.
    The forward-SDE noise is injected so both arrangements see identical eps."""
    from dmip import distributed as dd
    from dmip import losses as dl
    x, y, t = _dp_problem()
    B = x.shape[0]
    eps = torch.randn(B, 2, generator=torch.Generator().manual_seed(9))
    m, loss_fn = _dp_model_and_loss(kind)
    m.sde.to(DEV)

    def run(sl, bg, grad_out=None):
        xs, ys, ts, es = (v[sl].to(DEV) for v in (x, y, t, eps))
        if kind == "DSM":
            loss, _ = dl.dsm_fused(m, xs, ys, ts, es, batch_global=bg, grad_out=grad_out)
            return loss
        loss_fn.batch_global, loss_fn.grad_out = bg, grad_out
        try:
            loss, _ = loss_fn(m.sde, xs, ys, xs, ts, es, None, None)
        finally:
            loss_fn.batch_global, loss_fn.grad_out = 0, None
        return loss

    full = run(slice(0, B), 0)
    m.sde.a.zero_grad()
    full.backward()
    ref = torch.cat([p.grad.reshape(-1) for p in m.sde.a.parameters()]).clone()
    buckets, losses = [], []
    for r in range(2):
        s, c = dd.shard_range(B, r, 2)
        b = dd.GradBucket([m.sde.a])
        with torch.no_grad():
            losses.append(run(slice(s, s + c), B, b.grads).detach())
        buckets.append(b.grads.clone())
    got = buckets[0] + buckets[1]
    e_g = ((got - ref).abs().max() / ref.abs().max()).item()
    e_l = abs((losses[0] + losses[1]).item() - full.item()) / abs(full.item())
    return max(e_g / 2e-4, e_l / 1e-5), 1.0, dict(e_g=e_g, e_l=e_l)


def _dp_nccl_worker(rank, world, port, kind, ret):
    import os
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
    try:
        from dmip import distributed as dd
        x, y, t = _dp_problem()
        B = x.shape[0]
        m, loss_fn = _dp_model_and_loss(kind)          # same seed on every rank: identical weights
        m.sde.to(f"cuda:{rank}")
        opt = torch.optim.SGD(m.sde.a.parameters(), lr=0.0)     # lr 0: the step leaves the weights, the grads stay readable
        s, c = dd.shard_range(B, rank, world)
        dev = f"cuda:{rank}"
        torch.manual_seed(1234 + rank)
        loss, info = dd.train_step_data_parallel(m, opt, loss_fn, x[s:s + c].to(dev), y[s:s + c].to(dev), t[s:s + c].to(dev),
                                                 batch_global=B)
        flat = torch.cat([p.grad.reshape(-1) for p in m.sde.a.parameters()])
        ret[rank] = (loss.item(), flat.cpu(), {k: v.item() for k, v in info.items()})
    finally:
        dist.destroy_process_group()


def case_data_parallel_nccl(kind="DSM"):
    """Two real ranks (NCCL, one process per GPU; needs >= 2 GPUs): after train_step_data_parallel both ranks hold the SAME
    all-reduced gradient, and it equals the emulated sum of the two shards' gradients evaluated in this process on the
    same eps (seed 1234 + rank per shard) — the collective adds nothing but the sum."""
    import socket
    import torch.multiprocessing as mp
    from dmip import distributed as dd
    s_ = socket.socket()
    s_.bind(("127.0.0.1", 0))
    port = s_.getsockname()[1]
    s_.close()
    ctx = mp.get_context("spawn")
    with ctx.Manager() as mgr:
        ret = mgr.dict()
        procs = [ctx.Process(target=_dp_nccl_worker, args=(r, 2, port, kind, ret)) for r in range(2)]
        for p in procs:
            p.start()
        for p in procs:
            p.join(300)
            assert p.exitcode == 0, p.exitcode
        res = dict(ret)
    # the same two shards in this process, summed by hand
    from dmip.losses import fused_train_step
    x, y, t = _dp_problem()
    B = x.shape[0]
    m, loss_fn = _dp_model_and_loss(kind)
    m.sde.to(DEV)
    total, loss_sum = None, 0.0
    for r in range(2):
        s, c = dd.shard_range(B, r, 2)
        b = dd.GradBucket([m.sde.a])
        loss_fn.batch_global, loss_fn.grad_out = B, b.grads
        torch.manual_seed(1234 + r)
        with torch.no_grad():
            loss, _ = fused_train_step(m, loss_fn, x[s:s + c].to(DEV), y[s:s + c].to(DEV), t[s:s + c].to(DEV))
        loss_fn.batch_global, loss_fn.grad_out = 0, None
        total = b.grads.clone() if total is None else total + b.grads
        loss_sum += loss.item()
    total = total.cpu()
    e_same = (res[0][1] - res[1][1]).abs().max().item()
    e_g = ((res[0][1] - total).abs().max() / total.abs().max()).item()
    e_l = abs(res[0][0] - loss_sum) / abs(loss_sum)
    return max(e_same / 1e-12 if e_same > 0 else 0.0, e_g / 2e-4, e_l / 1e-5), 1.0, dict(e_same=e_same, e_g=e_g, e_l=e_l)


# ------------------------------------------------------------------------------------------- parity at BASELINE sizes
def case_loss_at_baseline_batch(kind, B=65536, chunk=4096):
    """BASELINE configs[1] size: linear CDE, batch 65,536 (2048 forward tiles over 148 SMs, split-K atomics over 144 CTAs,
    `batch_global` scaling), fused DSM / PINN(FPE exact, L1, ic L2) on the GPU against the CPU oracle in fp64, evaluated
    in chunks of 4096 rows and combined with the sum-of-means identity (SURVEY.md Q10): loss and every info mean within
    3e-4 relative, every parameter gradient within 3e-3 of its scale — the tolerances of the small fixtures."""
    from dmip import losses as dl
    from dmip.linear_problem import LinearForwardProblem
    from dmip.models.diffusion import CDE
    from oracle import losses as ol
    lin = LinearForwardProblem()
    g = torch.Generator().manual_seed(7)                           # SURVEY.md §8d config 2: x ~ N(0, I), seed 7
    x = torch.randn(B, 2, generator=g)
    y = lin(x) + 0.3 * torch.randn(B, 2, generator=g)
    t = torch.rand(B, 1, generator=g) * (1 - 2e-4) + 1e-4
    eps = torch.randn(B, 2, generator=g)
    ic = lin.score_posterior(x, y)
    params = make_params(0, 5, 2)
    m = CDE(2, 2, [512, 512, 512])
    m.sde.a.load_state_dict(state_dict_from_params(params))
    m.sde.to(DEV)
    kw = dict(lam=0.001, lam2=0.1, pde_loss="FPE", ic_metric="L2", pde_metric="L1")    # config_linear.yml:11-16
    xd, yd, td, ed = (v.to(DEV) for v in (x, y, t, eps))
    if kind == "DSM":
        loss, _ = dl.dsm_fused(m, xd, yd, td, ed)
        info = {}
    else:
        icd = ic.to(DEV)
        loss_fn = dl.PINNLoss(lambda xx, yy: icd, **kw)
        loss, info = loss_fn(m.sde, xd, yd, xd, td, ed, None, None)
    m.sde.a.zero_grad()
    loss.backward()
    got = [p.grad.detach().cpu().double() for p in m.sde.a.parameters()]
    # oracle: fp64, chunked
    p64 = [(W.double().requires_grad_(True), b.double().requires_grad_(True)) for W, b in params]
    tot, tinfo = 0.0, {}
    torch.set_num_threads(max(torch.get_num_threads(), 8))
    for s in range(0, B, chunk):
        sl = slice(s, s + chunk)
        a = [v[sl].double() for v in (x, y, t, eps)]
        if kind == "DSM":
            lc, ic_info = ol.dsm_loss(p64, "CDE", *a), {}
        else:
            lc, ic_info = ol.pinn_loss(p64, "CDE", *a, ic[sl].double(), **kw)
        w = (min(B, s + chunk) - s) / B
        (lc * w).backward()
        tot += lc.item() * w
        for k, v in ic_info.items():
            tinfo[k] = tinfo.get(k, 0.0) + v.item() * w
    err = abs(loss.item() - tot) / abs(tot)
    for k, v in info.items():
        err = max(err, abs(v.item() - tinfo[k]) / max(abs(tinfo[k]), 1e-12))
    ref = [q.grad for W, b in p64 for q in (W, b)]
    e_g = 0.0
    for a_, r_ in zip(got, ref):
        scale = r_.norm().item() / max(r_.numel() ** 0.5, 1.0)
        e_g = max(e_g, (a_ - r_).abs().max().item() / (3e-3 * scale + 3e-3 * r_.abs().max().item()))
    return max(err / 3e-4, e_g), 1.0, dict(loss=loss.item(), ref=tot, e_loss=err, e_grad=e_g)


def case_loss_repeats(kind, B=65536 + 37, reps=12):
    """Stand-in for compute-sanitizer racecheck (closed on this pool) on the cross-CTA protocol of the CTA-pair loss
    kernels: the same fused step, `reps` times on the same inputs, at a batch that leaves the last tile pair ragged (one
    CTA of the last cluster runs an empty tile).  Every repeat must give the loss and every gradient of the first one
    up to the reordering of fp32 atomics (3e-5 relative to each tensor's largest entry): an operand read before its rows
    were written, or a stale weight stage, would show as a wrong result, not as rounding."""
    from dmip import losses as dl
    from dmip.linear_problem import LinearForwardProblem
    from dmip.models.diffusion import CDE
    lin = LinearForwardProblem()
    g = torch.Generator().manual_seed(11)
    x = torch.randn(B, 2, generator=g)
    y = lin(x) + 0.3 * torch.randn(B, 2, generator=g)
    t = torch.rand(B, 1, generator=g) * (1 - 2e-4) + 1e-4
    eps = torch.randn(B, 2, generator=g)
    torch.manual_seed(3)
    m = CDE(2, 2, [512, 512, 512])
    m.sde.to(DEV)
    xd, yd, td, ed = (v.to(DEV) for v in (x, y, t, eps))
    icd = lin.score_posterior(x, y).to(DEV)
    loss_fn = dl.PINNLoss(lambda xx, yy: icd, lam=0.001, lam2=0.1, pde_loss="FPE", ic_metric="L2", pde_metric="L1")
    first, worst = None, 0.0
    for _ in range(reps):
        if kind == "DSM":
            loss, _ = dl.dsm_fused(m, xd, yd, td, ed)
        else:
            loss, _ = loss_fn(m.sde, xd, yd, xd, td, ed, None, None)
        m.sde.a.zero_grad()
        loss.backward()
        cur = [loss.detach().double().reshape(1)] + [p.grad.detach().double().clone() for p in m.sde.a.parameters()]
        if first is None:
            first = cur
            continue
        for a_, r_ in zip(cur, first):
            worst = max(worst, ((a_ - r_).abs().max() / r_.abs().max().clamp_min(1e-30)).item())
    ok = all(torch.isfinite(v).all().item() for v in first)
    return (worst if ok else float("inf")), 3e-5, dict(reps=reps, batch=B, loss=first[0].item())


def case_train_epoch_paths_agree(loss_name):
    """`train_epoch` with the fused optimizer step (the optimizer holds exactly the net's parameters) against the literal
    zero_grad / backward / step triple (taken when it holds anything else — here one extra parameter): same seeds, so
    the same t and noise draws; after an epoch of 6 batches of 1000 the parameters agree up to fp32 atomics, the
    returned loss and info dict too; and the fast path was the one that ran (p.grad aliases the gradient bucket)."""
    from dmip import losses as dl
    from dmip.linear_problem import LinearForwardProblem
    from dmip.models.diffusion import CDE
    lin = LinearForwardProblem()
    g = torch.Generator().manual_seed(21)
    x = torch.randn(6000, 2, generator=g)
    y = lin(x) + 0.3 * torch.randn(6000, 2, generator=g)
    xd, yd = x.to(DEV), y.to(DEV)

    def loader():
        for i in range(0, 6000, 1000):
            yield xd[i:i + 1000], yd[i:i + 1000]

    res = []
    for extra in (False, True):
        torch.manual_seed(4)
        m = CDE(2, 2, [512, 512, 512])
        params = list(m.sde.a.parameters())
        dummy = torch.nn.Parameter(torch.zeros(3, device=DEV))
        opt = torch.optim.Adam(params + ([dummy] if extra else []), lr=1e-3)
        if loss_name == "DSM":
            loss_fn = dl.DSMLoss()
        else:
            ic = lin.score_posterior(x, y).to(DEV)
            table = {}
            loss_fn = dl.PINNLoss(lambda xx, yy: ic[table.setdefault(xx.data_ptr(), len(table)) * 1000:][:1000],
                                  lam=0.001, lam2=0.1, pde_loss="FPE", ic_metric="L2", pde_metric="L1")
        torch.manual_seed(9)
        loss, info = m.train_epoch(opt, loss_fn, loader)
        fast = hasattr(m, "_grad_bucket") and params[0].grad is not None and \
            params[0].grad.data_ptr() == m._grad_bucket.flat.data_ptr()
        res.append((loss.item(), info, [p.detach().clone() for p in params], fast))
    (l0, i0, p0, f0), (l1, i1, p1, f1) = res
    err = abs(l0 - l1) / abs(l1)
    for k in i1:
        err = max(err, abs(i0[k] - i1[k]) / max(abs(i1[k]), 1e-12))
    for a_, b_ in zip(p0, p1):
        err = max(err, ((a_ - b_).abs().max() / b_.abs().max()).item())
    ok = f0 and not f1 and set(i0) == set(i1) and all(isinstance(v, float) for v in i0.values())
    return (err if ok else float("inf")), 2e-5, dict(loss_fast=l0, loss_literal=l1, fast_path=(f0, f1))


def case_sample_t_device():
    """dmip_sample_t against the host mirror (dmip.sdes.vp_truncated_inverse_cdf + the eps handling of
    models/diffusion.py:48-58) on the same uniforms, including u = 0, the kink at t_epsilon and u -> 1; and
    `model.sample_t` on a CUDA batch: shape, dtype, leaf with requires_grad, range (eps, T]."""
    import ctypes as C
    from dmip import _lib, sdes
    from dmip.models.diffusion import CDE
    sde = sdes.VariancePreservingSDE()
    u = torch.cat([torch.tensor([0.0, 1e-7, 1e-4, 1.0 - 6e-8]), torch.rand(100000, generator=torch.Generator().manual_seed(5))])
    worst = 0.0
    for debias in (True, False):
        ud = u.to(DEV)
        sde.sample_t_device([1], DEV)                                   # binds the entry point
        L = _lib.require_gpu()
        t = torch.empty_like(ud)
        _lib.check(L.dmip_sample_t(ud.data_ptr(), t.data_ptr(), ud.numel(), int(debias), float(sde.beta_min),
                                   float(sde.beta_max), float(sde.t_epsilon), float(sde.T), 1e-4, _lib.stream_ptr()))
        if debias:
            ref = sdes.vp_truncated_inverse_cdf(u.double(), sde.beta_min, sde.beta_max, sde.t_epsilon, sde.T) + 1e-4
            ref = torch.where(ref.float() > sde.T, ref - 1e-4, ref)
        else:
            ref = 1e-4 + u.double() * sde.T
            ref = torch.where(ref.float() > sde.T, torch.full_like(ref, sde.T - 1e-4), ref)
        worst = max(worst, (t.cpu().double() - ref).abs().max().item())
    m = CDE(2, 2, [512, 512, 512])
    x = torch.randn(1000, 2, device=DEV)
    tt = m.sample_t(x)
    ok = (tt.shape == (1000, 1) and tt.dtype == torch.float32 and tt.is_cuda and tt.requires_grad and tt.is_leaf
          and tt.min().item() > 1e-4 and tt.max().item() <= 1.0)
    return (worst if ok else float("inf")), 2e-7, dict(worst=worst)


def case_sampler_trained_1000_steps(precision):
    """Trained linear CDE at S = 1000 steps (5x the reference default: bf16 rounding accumulates 5x longer), N = 512,
    the keyed Philox stream injected, against the CPU oracle sampler on the same noise: fp32 5e-4, bf16 1e-2 max abs
    with |mean shift| <= 3e-3 and |std ratio - 1| <= 5e-3 (SURVEY.md §8d)."""
    fx = load_golden("trained_cde_linear")
    params = on.params_from_state_dict({f"{k}.{n}": fx[f"{k}_{n}"] for k in (0, 3, 5, 7) for n in ("weight", "bias")})
    m = trained_model()
    N, S, seed = 512, 1000, 4242
    y = torch.tensor([0.4, -0.7])
    gidx = np.arange(N)
    x0 = torch.from_numpy(oracle.philox.normals(gidx, oracle.philox.STEP_INIT, 0, 2, seed))
    noise = torch.from_numpy(np.stack([oracle.philox.normals(gidx, i, 0, 2, seed) for i in range(S)]))
    with torch.no_grad():
        ref = osamp.em_sampler_cde(params, y, x0, noise, S)
    out = torch.from_numpy(m(y, num_samples=N, num_steps=S, precision=precision, injected=dict(x0=x0, noise=noise)))
    out_p = torch.from_numpy(m(y, num_samples=N, num_steps=S, precision=precision, seed=seed))     # in-kernel Philox
    err = max((out - ref).abs().max().item(), (out_p - ref).abs().max().item())
    tol = 5e-4 if precision == "fp32" else 1e-2
    dmean = (out.mean(0) - ref.mean(0)).abs().max().item()
    rstd = (out.std(0) / ref.std(0) - 1).abs().max().item()
    if precision == "bf16" and (dmean > 3e-3 or rstd > 5e-3):
        err = max(err, 1.0)
    return err, tol, dict(out=out, ref=ref, dmean=dmean, rstd=rstd)


def case_philox_equals_injected(kind, precision):
    """CDiffE (in-kernel re-diffusion stream of y, Philox stream 1) and DPS (two-net pass): the kernel's own Philox
    draws must reproduce the run fed with the numpy mirror of the same keyed streams (oracle/philox.py), as the CDE
    cases already check.  Scatterometry shapes (xdim 3, ydim 23), untrained nets, S = 10: relative to max|x|, fp32 1e-4
    (transcendental intrinsics differ from numpy by ~1e-6 per draw and the untrained dynamics amplify), bf16 2e-3."""
    xdim, ydim, N, S, seed, base = 3, 23, 300, 10, 991, 5000
    m = _model(kind, xdim, ydim, (512, 512, 512), 61)
    y = torch.randn(ydim, generator=torch.Generator().manual_seed(2))
    gidx = np.arange(N) + base
    inj = dict(x0=torch.from_numpy(oracle.philox.normals(gidx, oracle.philox.STEP_INIT, 0, xdim, seed)),
               noise=torch.from_numpy(np.stack([oracle.philox.normals(gidx, i, 0, xdim, seed) for i in range(S)])))
    if kind == "CDiffE":
        inj["ynoise"] = torch.from_numpy(np.stack([oracle.philox.normals(gidx, i, 1, ydim, seed) for i in range(S)]))
    a = m(y, num_samples=N, num_steps=S, precision=precision, seed=seed, gidx_base=base, return_tensor=True)
    b = m(y, num_samples=N, num_steps=S, precision=precision, injected=inj, return_tensor=True)
    err = ((a - b).abs().max() / b.abs().max()).item()
    return err, (1e-4 if precision == "fp32" else 2e-3), dict(out=a.cpu(), ref=b.cpu())


def case_batched_observations_variant(kind):
    """y of shape (n_obs, ydim) for CDiffE and DPS: all observations in ONE launch == one call per observation with the
    matching global-index offset, bit for bit (BASELINE configs[3]: observations are the sharded unit)."""
    xdim, ydim = 3, 23
    m = _model(kind, xdim, ydim, (512, 512, 512), 62)
    ys = torch.randn(3, ydim, generator=torch.Generator().manual_seed(5))
    N, S, seed = 200, 8, 7
    batched = m(ys, num_samples=N, num_steps=S, seed=seed, return_tensor=True)
    assert batched.shape == (3, N, xdim)
    err = 0.0
    for o in range(3):
        single = m(ys[o], num_samples=N, num_steps=S, seed=seed, gidx_base=o * N, return_tensor=True)
        err = max(err, (single - batched[o]).abs().max().item())
    # and through the public sharding helper: observations split over ranks (world size 1 here -> all of them)
    from dmip.distributed import sample_sharded
    one = sample_sharded(m, ys, num_samples=N, num_steps=S, seed=seed, shard='observations')
    err = max(err, (one.view(3, N, xdim) - batched).abs().max().item())
    return err, 0.0, {}


_SCAT_MODELS = {}


def _trained_scat_model(kind):
    """A briefly DSM-trained scatterometry model (CDiffE: joint score of [x, y]; DPS: PosteriorLoss on both nets), so
    that the reverse SDE contracts and sample statistics are meaningful; cached per process."""
    if kind in _SCAT_MODELS:
        return _SCAT_MODELS[kind]
    from dmip import losses as dl
    from dmip.models.diffusion import CDiffE, PosteriorDiffusionEstimator
    fm, _ = _surrogate_module()
    torch.manual_seed(0)
    X = torch.rand(8000, 3, device=DEV) * 2 - 1
    with torch.no_grad():
        fX = fm(X)
        Y = fX + 0.01 * torch.randn_like(fX) + 0.2 * fX * torch.randn_like(fX)
    loader = lambda: ((X[i:i + 1000], Y[i:i + 1000]) for i in range(0, 8000, 1000))
    if kind == "CDiffE":
        m = CDiffE(3, 23, [512, 512, 512])
        m.sde.to(DEV)
        opt = torch.optim.Adam(m.sde.a.parameters(), lr=1e-3)
        for _ in range(40):
            m.train_epoch(opt, dl.DSMLoss(), loader)
    else:
        m = PosteriorDiffusionEstimator(3, 23, [512, 512, 512])
        m.sde.to(DEV)
        opt = torch.optim.Adam(m.sde.a.parameters(), lr=1e-3)
        loss_fn = m.loss_fn(fm, 0.2, 0.01, lam=1e-4)
        for _ in range(40):
            m.train_epoch(opt, loss_fn, loader)
    m.sde.eval()
    _SCAT_MODELS[kind] = (m, fm, Y)
    return _SCAT_MODELS[kind]


def case_scat_statistics(kind):
    """Posterior statistics of the bf16 tensor-core sampler against the fp32 kernel for a trained scatterometry CDiffE /
    DPS model (models/diffusion.py:158-180, nets.py:155-157): 65,536 particles, 200 steps, same Philox key.
    |mean shift| <= 5e-3 and |std ratio - 1| <= 1e-2 per coordinate, and the reference's own metric — the 75-bin histogram
    KL on [-1.2, 1.2]^3 (main_diffusion_scatterometry.py:72-101) — between the two precisions <= 1.5 x the KL between two
    independent fp32 runs (SURVEY.md §8d statistical tolerance)."""
    from dmip import metrics as dmet
    m, fm, Y = _trained_scat_model(kind)
    y = Y[17].cpu()
    N, S = 65536, 200
    sets = {k: m(y, num_samples=N, num_steps=S, precision=p, seed=s, return_tensor=True)
            for k, (p, s) in dict(lo=("bf16", 31), hi=("fp32", 31), hi2=("fp32", 32), lo2=("bf16", 33)).items()}
    finite = all(bool(torch.isfinite(v).all()) for v in sets.values())
    dmean = (sets["lo"].mean(0) - sets["hi"].mean(0)).abs().max().item()
    rstd = (sets["lo"].std(0) / sets["hi"].std(0) - 1).abs().max().item()
    bins, rng = (75, 75, 75), ((-1.2, 1.2),) * 3
    h = {k: dmet.histogramdd(v, bins, rng) for k, v in sets.items()}
    kl_new = float(dmet.hist_kl(h["hi"], h["lo2"]))
    kl_ref = float(dmet.hist_kl(h["hi"], h["hi2"]))
    inside = float(h["hi"].sum().item()) / N
    err = max(dmean / 5e-3, rstd / 1e-2, kl_new / (1.5 * kl_ref) if kl_ref > 0 else 0.0, 0.0 if finite else 2.0,
              0.0 if inside > 0.5 else 2.0)
    return err, 1.0, dict(dmean=dmean, rstd=rstd, kl_new=kl_new, kl_ref=kl_ref, inside=inside)


# ------------------------------------------------------------------------------------------- VE-SDE / predictor–corrector (N4)
def case_pc_sampler(kind, sde_kind, n_corr, precision):
    """VE-SDE and Langevin-corrector modes of the fused sampler (no upstream counterpart: parity unpinned, SURVEY.md §8f N4)
    against the oracle restatement oracle/ve.py — which with the VP-SDE and no corrector IS the pinned reference sampler
    (tests/test_oracle_golden.py).  Injected noise, scatterometry shapes, untrained nets, S = 8 steps (x (1 + n_corr)
    sub-steps): relative to max|x|, fp32 2e-5, bf16 3e-3; and the in-kernel Philox stream keyed by the sub-step index must
    reproduce the run fed with its numpy mirror (fp32 1e-4, bf16 2e-3)."""
    from dmip import sdes
    from dmip.models.diffusion import CDE, CDiffE, PosteriorDiffusionEstimator
    from oracle import ve
    xdim, ydim, N, S, seed, snr = 3, 23, 200, 8, 77, 0.16
    hidden = (512, 512, 512)
    base = sdes.VarianceExplodingSDE(sigma_min=0.05, sigma_max=4.0) if sde_kind == "VE" else None
    osde = ve.VE(0.05, 4.0) if sde_kind == "VE" else ve.VP()
    if kind == "CDE":
        m = CDE(xdim, ydim, list(hidden), base_sde=base)
        p = make_params(71, xdim + ydim + 1, xdim, hidden)
        m.sde.a.load_state_dict(state_dict_from_params(p))
        net, variant = ve.net_fn("CDE", p), "CDE"
    elif kind == "CDiffE":
        m = CDiffE(xdim, ydim, list(hidden), base_sde=base)
        p = make_params(72, xdim + ydim + 1, xdim + ydim, hidden)
        m.sde.a.load_state_dict(state_dict_from_params(p))
        net, variant = ve.net_fn("CDiffE", p), "CDiffE"
    else:
        m = PosteriorDiffusionEstimator(xdim, ydim, list(hidden), base_sde=base)
        p2, p = make_params(73, xdim + 1, xdim, hidden), make_params(173, xdim + ydim + 1, xdim, hidden)
        m.sde.a.prior_net.load_state_dict(state_dict_from_params(p2))
        m.sde.a.likelihood_net.load_state_dict(state_dict_from_params(p))
        net, variant = ve.net_fn("DPS", p, p2), "DPS"
    m.sde.to(DEV)
    y = torch.randn(ydim, generator=torch.Generator().manual_seed(3))
    std0 = 4.0 if sde_kind == "VE" else 1.0
    n_sub = S * (1 + n_corr)
    gidx = np.arange(N)
    x0 = torch.from_numpy(oracle.philox.normals(gidx, oracle.philox.STEP_INIT, 0, xdim, seed))
    noise = torch.from_numpy(np.stack([oracle.philox.normals(gidx, u, 0, xdim, seed) for u in range(n_sub)]))
    inj = dict(x0=x0, noise=noise)
    ynoise = None
    if kind == "CDiffE":
        ynoise = torch.from_numpy(np.stack([oracle.philox.normals(gidx, u, 1, ydim, seed) for u in range(n_sub)]))
        inj["ynoise"] = ynoise
    with torch.no_grad():
        ref = ve.pc_sampler(net, variant, y, x0 * std0, noise, S, osde, n_corr=n_corr, snr=snr, ynoise=ynoise)
    kw = dict(num_samples=N, num_steps=S, std=std0, precision=precision, n_corrector=n_corr, snr=snr)
    out = torch.from_numpy(m(y, injected=inj, **kw))
    out_p = torch.from_numpy(m(y, seed=seed, **kw))
    scale = ref.abs().max().item()
    e_inj = (out - ref).abs().max().item() / scale
    e_phx = (out_p - out).abs().max().item() / scale
    t_inj, t_phx = (2e-5, 1e-4) if precision == "fp32" else (3e-3, 2e-3)
    return max(e_inj / t_inj, e_phx / t_phx), 1.0, dict(e_inj=e_inj, e_phx=e_phx, out=out, ref=ref)


def case_ve_trained_posterior():
    """A VE-SDE CDE trained on the linear problem with a host-side DSM loop cannot use the fused (VP-only) losses, so the
    statistical check of the VE / corrector samplers uses the ANALYTIC score of the linear-Gaussian posterior instead:
    the perturbed posterior N(m, C + sigma(t)^2 I) has score -(C + sigma^2 I)^-1 (x - m), which a [512,512,512] net
    cannot represent exactly — so the check is self-consistency: bf16 vs fp32 kernels on the same Philox key, with and
    without the corrector (mean shift <= 2e-2 sigma-units, std ratio within 2e-2), on an untrained net scaled down to a
    contraction.  (Documented limitation: no trained VE model exists upstream or here.)"""
    from dmip import sdes
    from dmip.models.diffusion import CDE
    torch.manual_seed(0)
    m = CDE(2, 2, [512, 512, 512], base_sde=sdes.VarianceExplodingSDE(sigma_min=0.05, sigma_max=2.0))
    with torch.no_grad():
        for p in m.sde.a.parameters():
            p.mul_(0.5)
    m.sde.to(DEV)
    y = torch.tensor([0.4, -0.7])
    worst = 0.0
    for nc in (0, 1):
        lo = m(y, num_samples=32768, num_steps=100, std=2.0, precision="bf16", seed=5, n_corrector=nc)
        hi = m(y, num_samples=32768, num_steps=100, std=2.0, precision="fp32", seed=5, n_corrector=nc)
        assert np.isfinite(lo).all() and np.isfinite(hi).all()
        dmean = float(np.abs(lo.mean(0) - hi.mean(0)).max() / hi.std(0).max())
        rstd = float(np.abs(lo.std(0) / hi.std(0) - 1).max())
        worst = max(worst, dmean / 2e-2, rstd / 2e-2)
    return worst, 1.0, {}


# ------------------------------------------------------------------------------------------- evaluate-loop parity (N2)
def case_evaluate_parity(problem):
    """dmip.evaluation against tables produced by the reference's OWN evaluate loops (main_diffusion_linear.py:53-137,
    main_diffusion_scatterometry.py:40-124) on stored sample sets (oracle/make_golden.py §5c: the reference code ran with
    its sampler / posterior draws / ground-truth files replaced by players of the fixture arrays).  KL2 / KL_reverse
    1e-9 relative (bit-exact counts, float64 KL), NLL columns 1e-5, score MSE 1e-4 (fp32 score net)."""
    from dmip import evaluation
    from dmip.linear_problem import LinearForwardProblem
    from dmip.models.diffusion import CDE
    from dmip.utils_scatterometry import make_score_posterior
    fx = load_golden("eval_" + problem, dtype=torch.float64)
    xp, xt = fx["x_pred"].float(), fx["x_true"].float()
    sets = lambda x: [x[:, j].contiguous().to(DEV) for j in range(x.shape[1])]
    if problem == "linear":
        m = trained_model()
        m.sde.a.precision = "fp32"
        table = evaluation.linear_metrics(m, fx["ys"].float(), LinearForwardProblem(), sets(xp), sets(xt))
        cols = dict(KL2=1e-9, NLL_true=1e-5, NLL_diffusion=1e-5, MSE=1e-4)
    else:
        fm, _ = _surrogate_module()
        m = CDE(3, 23, [512, 512, 512])
        m.sde.a.load_state_dict(state_dict_from_params(make_params(95, 27, 3)))
        m.sde.to(DEV)
        m.sde.a.precision = "fp32"
        sp = make_score_posterior(fm, dict(a=0.2, b=0.01, lambd_bd=1000))
        table = evaluation.scatterometry_metrics(m, fx["ys"].float(), fm, sets(xp), sets(xt), sp, 0.2, 0.01, 1000)
        cols = dict(KL2=1e-9, KL_reverse=1e-9, NLL_mcmc=1e-5, NLL_diffusion=1e-5, MSE=1e-4)
    worst, detail = 0.0, {}
    for c, tol in cols.items():
        ref = fx[c].numpy()
        e = float(np.max(np.abs(table[c] - ref) / np.maximum(np.abs(ref), 1e-12)))
        detail[c] = e
        worst = max(worst, e / tol)
    return worst, 1.0, detail


# ------------------------------------------------------------------------------------------- bounds check (sanitizer stand-in)
def case_guarded_buffers():
    """compute-sanitizer is closed on this GPU pool (profiles/r02_compute_sanitizer_closed.txt).  Stand-in bounds check:
    with DMIP_GUARD=1 every output / scratch buffer handed to the library is wrapped in 4 KB canaries that are verified
    after the call (dmip._lib.Guarded) — the packed workspace of the tcgen05 loss path (images, stashes, adjoints), the
    flat gradient, the loss scalars and the sampler's output, over ragged batch sizes (tile tails, masked cluster CTAs)
    and all three sampler variants; the surrogate kernels' outputs and workspace (weight images) at ragged row counts."""
    import os
    from dmip import losses as dl
    from dmip.models.diffusion import CDE
    os.environ["DMIP_GUARD"] = "1"
    try:
        torch.manual_seed(0)
        m = CDE(2, 2, [512, 512, 512])
        m.sde.to(DEV)
        for path in ("tc", "ffma"):
            os.environ["DMIP_LOSS_PATH"] = path
            for B in (1, 7, 8, 63, 64, 65, 129, 1000, 2963):
                x, y, t = _dp_problem(B)
                xd, yd, td = x.to(DEV), y.to(DEV), t.to(DEV)
                eps = torch.randn(B, 2, device=DEV)
                dl.dsm_fused(m, xd, yd, td, eps)
                for kw in (dict(pde_loss="FPE"), dict(pde_loss="cScoreFPE")):
                    fn = dl.PINNLoss(lambda xx, yy: -xx, lam=0.01, lam2=0.1, ic_metric="L2", pde_metric="L1", **kw)
                    fn(m.sde, xd, yd, xd, td, eps, None, None)
                dl.DSM_PDELoss(lam=0.1, pde_loss="FPE", pde_metric="L1")(m.sde, xd, yd, xd, td, eps, None, None)
        os.environ.pop("DMIP_LOSS_PATH", None)
        for kind in ("CDE", "CDiffE", "Posterior"):
            ms = _model(kind, 3, 23, (512, 512, 512), 9)
            yv = torch.randn(23)
            for N in (1, 127, 129, 300):
                for prec in ("bf16", "fp32"):
                    ms(yv, num_samples=N, num_steps=3, precision=prec, seed=1, n_corrector=1)
        # K4, both kernel families: ragged row counts, with and without the optional outputs, one observation for all rows
        from dmip import utils_scatterometry as us
        fm, _ = _surrogate_module()
        fxs = load_golden("scat_energy")
        for path in ("tc", "ffma"):
            _surrogate_path(path)
            for n in (1, 127, 128, 129, 512):
                xs, ysn = fxs["x"][:n].to(DEV), fxs["y"][:n].to(DEV)
                us.surrogate_call(fm, xs, ysn, 0.2, 0.01, 1000.0, want_fx=True)
                us.surrogate_call(fm, xs, ysn[:1], 0.2, 0.01, 1000.0, mode=us.SURR_LIK_VJP)
        _surrogate_path("tc")
    finally:
        os.environ.pop("DMIP_GUARD", None)
        os.environ.pop("DMIP_SURROGATE_PATH", None)
        os.environ.pop("DMIP_LOSS_PATH", None)
    return 0.0, 0.5, {}


# ------------------------------------------------------------------------------------------- documented boundary deviations
def case_boundary_deviations():
    """INTEGRATION.md "deviations": (1) ScoreFPELoss.forward / ConditionalScoreFPELoss.forward raise (the residual needs the
    net, not a detached score tensor); (2) PINNLoss / DSM_PDELoss called with the reference's full argument list validate
    that `diffused_samples` is the x_t the kernels re-derive — a different x_t raises instead of silently giving another
    loss; a consistent one gives the same loss as the internal call; (3) autograd through MLP.forward warns (eager torch
    path) and still returns correct gradients; (4) `train_step_data_parallel` leaves no `batch_global` behind."""
    import warnings
    from dmip import distributed as dd, losses as dl, nets as dnets
    from dmip.models.diffusion import CDE
    torch.manual_seed(0)
    m = CDE(2, 2, [512, 512, 512])
    m.sde.to(DEV)
    x, y, t = (v.to(DEV) for v in _dp_problem(256))
    ok = True
    for cls in (dl.ScoreFPELoss, dl.ConditionalScoreFPELoss):
        try:
            cls().forward(*([x] * (4 if cls is dl.ScoreFPELoss else 6)))
            ok = False
        except RuntimeError:
            pass
    loss_fn = dl.PINNLoss(lambda xx, yy: -xx, lam=0.001, lam2=0.1, pde_loss="FPE", ic_metric="L2", pde_metric="L1")
    x_t, eps, std, g = m.sde.base_sde.sample(t, x, return_noise=True)          # the reference's call sequence
    full, _ = loss_fn(m.sde, x, y, x_t, t, eps, std, g)
    short, _ = loss_fn(m.sde, x, y, x, t, eps, None, None)
    ok = ok and abs(full.item() - short.item()) <= 1e-6 * abs(short.item())
    try:
        loss_fn(m.sde, x, y, x_t + 0.1, t, eps, std, g)
        ok = False
    except ValueError:
        pass
    dnets._WARNED_EAGER[0] = False
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        tt = t.clone().requires_grad_(True)
        out = m.sde.a(x, y, tt)                     # [512,512,512]: autograd on the library's own kernels, no warning
        out.sum().backward()
        ok = ok and not w and tt.grad is not None
        small = dnets.MLP(5, 2, [64, 64], torch.nn.Tanh()).to(DEV)      # other widths: torch module chain, says so
        small(x, y, t.clone().requires_grad_(True)).sum().backward()
        ok = ok and any("autograd is recording" in str(i.message) for i in w)
    opt = torch.optim.SGD(m.sde.a.parameters(), lr=0.0)
    dd.train_step_data_parallel(m, opt, loss_fn, x, y, t)
    ok = ok and getattr(loss_fn, "batch_global", 0) == 0 and getattr(loss_fn, "grad_out", None) is None
    return (0.0 if ok else 1.0), 0.5, {}


# ------------------------------------------------------------------------------------------- autograd through the score net
def case_mlp_autograd(which):
    """`loss.backward()` of a user-written loss through MLP / MLP2.forward: the library's own forward-with-stash and
    backward kernels (dmip_mlp_forward_stash / dmip_mlp_backward, tcgen05, bf16x3) against torch's autograd through the
    plain module chain in fp64: outputs 2e-5 of their scale, every parameter gradient and the gradients w.r.t. x, y and t
    3e-4 of theirs.  Ragged batch (tile tail + masked cluster CTA)."""
    from dmip import nets as dnets
    torch.manual_seed(1)
    n = 333
    if which == "cde_linear":
        net, xd, cd = dnets.MLP(5, 2, [512, 512, 512], torch.nn.Tanh()), 2, 2
    elif which == "cdiffe_scat":
        net, xd, cd = dnets.MLP(27, 26, [512, 512, 512], torch.nn.Tanh()), 26, 0
    else:
        net, xd, cd = dnets.MLP2(4, 3, [512, 512, 512], torch.nn.Tanh()), 3, 0
    net.to(DEV)
    x = torch.randn(n, xd, device=DEV, requires_grad=True)
    y = torch.randn(n, cd, device=DEV, requires_grad=True) if cd else None
    t = torch.rand(n, 1, device=DEV, requires_grad=True)
    wgt = torch.randn(n, net.output_dim, device=DEV)

    def call(mod, xx, yy, ttt):
        if which == "mlp2":
            return mod(xx, ttt)
        return mod(xx, yy if yy is not None else torch.Tensor([]).to(DEV), ttt)

    out = call(net, x, y, t)
    (out * wgt).sum().backward()
    got = [out.detach()] + [p.grad.clone() for p in net.parameters()] + [v.grad.clone() for v in (x, y, t) if v is not None]
    # fp64 reference through the plain module chain
    import copy
    ref_net = copy.deepcopy(net).double()
    xr, tr = x.detach().double().requires_grad_(True), t.detach().double().requires_grad_(True)
    yr = y.detach().double().requires_grad_(True) if cd else None
    parts = [xr] + ([yr] if cd else []) + [tr]
    ro = torch.nn.Sequential.forward(ref_net, torch.cat(parts, 1))
    (ro * wgt.double()).sum().backward()
    ref = [ro.detach()] + [p.grad for p in ref_net.parameters()] + [v.grad for v in (xr, yr, tr) if v is not None]
    worst = 0.0
    for i, (a, b) in enumerate(zip(got, ref)):
        e = ((a.double() - b).abs().max() / b.abs().max()).item()
        worst = max(worst, e / (2e-5 if i == 0 else 3e-4))
    return worst, 1.0, {}


def case_graphed_steps_of_successive_models():
    """Three models in one process, each with a captured training step (eager Adam, capturable Adam, eager Adam): the
    capture of a later model must not be invalidated by the collection of an earlier model's graph (GraphedTrainStep
    keeps the garbage collector out of the capture) — the config0 bench line's loop.  Every epoch must lower the loss."""
    from dmip import losses as dl
    from dmip.models.diffusion import CDiffE
    worst = 0.0
    for capturable in (False, True, False):
        torch.manual_seed(0)
        model = CDiffE(2, 2, [512, 512, 512])
        model.sde.to(DEV)
        opt = torch.optim.Adam(model.sde.a.parameters(), lr=1e-3, capturable=capturable)
        g = torch.Generator().manual_seed(2)
        x = torch.randn(4000, 2, generator=g).to(DEV)
        y = (x + 0.3 * torch.randn(4000, 2, generator=g).to(DEV))
        loader = lambda: ((x[i:i + 1000], y[i:i + 1000]) for i in range(0, 4000, 1000))
        losses = [float(model.train_epoch(opt, dl.DSMLoss(), loader, graph=True)[0]) for _ in range(6)]
        captured = model.__dict__.get('_graphed_step') is not None
        worst = max(worst, 0.0 if (captured and losses[-1] < losses[0] and all(np.isfinite(losses))) else 1.0)
    return worst, 0.0, {}


# ------------------------------------------------------------------------------------------- fused losses: shape sweep
# The golden fixtures pin the fused losses at d in {2, 3, 26} and tile-aligned batches.  These cases run the public loss
# classes at any state dimension, net shape and batch, against the fp64 oracle evaluated in-process (oracle/losses.py,
# itself checked against a literal autograd statement at these shapes by tests/test_loss_oracle_shapes.py).
_SWEEP_REF = {}                 # oracle results of the last few (case, batch) keys: the tc and ffma runs share them


def _sweep_problem(model_kind, xdim, ydim, B, seed):
    """x, y ~ N(0, I); t ~ U[1e-4, 1 - 1e-4]; eps ~ N(0, I) (B, d); ic target ~ N(0, I) (B, xdim); probe +-1 (B, d)"""
    d = xdim if model_kind == "CDE" else xdim + ydim
    g = torch.Generator().manual_seed(1000 * seed + B)
    x = torch.randn(B, xdim, generator=g)
    y = torch.randn(B, ydim, generator=g)
    t = torch.rand(B, 1, generator=g) * (1 - 2e-4) + 1e-4
    eps = torch.randn(B, d, generator=g)
    ic = torch.randn(B, xdim, generator=g)
    probe = torch.randint(0, 2, (B, d), generator=g).float() * 2 - 1
    return x, y, t, eps, ic, probe


def _sweep_model(model_kind, xdim, ydim, hidden, seed):
    from dmip.models.diffusion import CDE, CDiffE
    d = xdim if model_kind == "CDE" else xdim + ydim
    params = make_params(seed, xdim + ydim + 1, d, hidden)
    m = (CDE if model_kind == "CDE" else CDiffE)(xdim, ydim, list(hidden))
    m.sde.a.load_state_dict(state_dict_from_params(params))
    m.sde.to(DEV)
    return m, params


def _sweep_library(m, model_kind, kind, kw, x, y, t, eps, ic, probe):
    """one fused forward+backward through the public classes -> (loss, info, parameter gradients, kernel launches)"""
    from dmip import losses as dl
    xd, yd, td, ed, icd, vd = (v.to(DEV) for v in (x, y, t, eps, ic, probe))
    info = {}
    if kind == "DSM":
        loss, launches = dl.dsm_fused(m, xd, yd, td, ed)
    else:
        if kind == "DSM_PDE":
            loss_fn = dl.DSM_PDELoss(**kw)
        else:
            loss_fn = (dl.PINNLoss if kind == "PINN" else dl.PINNLoss2)(lambda xx, yy: icd, **kw)
        loss_fn.probe = vd
        z = xd if model_kind == "CDE" else torch.cat([xd, yd], 1)
        loss, info = loss_fn(m.sde, xd, yd, z, td, ed, None, None)
        launches = loss_fn.last_launch_count
    m.sde.a.zero_grad()
    loss.backward()
    grads = [p.grad.detach().cpu().double() for p in m.sde.a.parameters()]
    return loss.item(), {k: v.item() for k, v in info.items()}, grads, launches


def _sweep_reference(key, params, model_kind, kind, kw, x, y, t, eps, ic, probe):
    """fp64 oracle: (loss, info, parameter gradients); 'exact' and 'exact_adjoint' share one entry"""
    from oracle import losses as ol
    if key in _SWEEP_REF:
        return _SWEEP_REF[key]
    torch.set_num_threads(max(torch.get_num_threads(), 8))
    kw = dict(kw)
    div = kw.pop("divergence_method", "exact")
    v = probe.double() if div in ("hutchinson", "approx", "approximate") else None
    p64 = [(W.double().requires_grad_(True), b.double().requires_grad_(True)) for W, b in params]
    a = [u.double() for u in (x, y, t, eps)]
    if kind == "DSM":
        loss, info = ol.dsm_loss(p64, model_kind, *a), {}
    elif kind == "DSM_PDE":
        loss, info = ol.dsm_pde_loss(p64, model_kind, *a, probe=v, **kw)
    else:
        fn = ol.pinn_loss if kind == "PINN" else ol.pinn2_loss
        loss, info = fn(p64, model_kind, *a, ic.double(), probe=v, **kw)
    loss.backward()
    ref = (loss.item(), {k: u.item() for k, u in info.items()}, [q.grad for W, b in p64 for q in (W, b)])
    while len(_SWEEP_REF) >= 4:
        _SWEEP_REF.pop(next(iter(_SWEEP_REF)))
    _SWEEP_REF[key] = ref
    return ref


def _sweep_errors(got, ref, loss_rtol):
    """max(loss / info relative error / loss_rtol, worst parameter-gradient error / (3e-3 (rms(ref) + max|ref|))):
    the criteria of case_loss_at_baseline_batch, <= 1 passes"""
    e_loss = abs(got[0] - ref[0]) / max(abs(ref[0]), 1e-6)
    for k, r in ref[1].items():
        e_loss = max(e_loss, abs(got[1][k] - r) / max(abs(r), 1e-6))
    e_g = 0.0
    for a_, r_ in zip(got[2], ref[2]):
        scale = r_.norm().item() / max(r_.numel() ** 0.5, 1.0) + r_.abs().max().item()
        e_g = max(e_g, (a_ - r_).abs().max().item() / max(3e-3 * scale, 1e-30))
    return max(e_loss / loss_rtol, e_g), e_loss, e_g


def _l1_margin(params, model_kind, kind, kw, x, y, t, eps, ic, probe):
    """Smallest |r| / max|r| over the residuals r a loss takes the L1 norm of (PDE residual, initial-condition difference).
    d|r|/dr jumps from -1 to 1 at r = 0: where fp32 rounding can flip the sign of r, the kernels' gradient and the fp64
    one legitimately differ by a whole term, and a one-sample batch then misses by several times the tolerance (seen at
    CDiffE 2 + 61, Hutchinson, B = 1: |R_7| = 2e-7 against a median |R| of 0.15).  The sweep redraws such a problem."""
    from oracle import losses as ol, nets as onets, vp
    p64 = [(W.double(), b.double()) for W, b in params]
    x, y, t, eps, ic = (u.double() for u in (x, y, t, eps, ic))
    pde = kw.get("pde_loss", "FPE")
    pde_metric = ("L1" if pde == "FPE" else "L2") if kind == "PINN2" else kw.get("pde_metric", "L1")
    res = []
    if kind in ("PINN", "PINN2") and kw.get("ic_metric", "L1") == "L1":
        t0 = torch.zeros_like(t)
        res.append(onets.mlp(p64, x, y, t0)[:, :x.shape[1]] / vp.beta(t0) ** 0.5 - ic)
    if kind != "DSM" and pde_metric == "L1":
        z0, cond, z_t, std = ol._split(model_kind, x, y, t, eps)
        hutch = kw.get("divergence_method", "exact") in ("hutchinson", "approx", "approximate")
        terms = ol.score_and_fpe_terms(p64, z_t, cond, t, z0, eps, need_space=(pde == "FPE"),
                                       probe=probe.double() if hutch else None)
        if pde == "FPE":
            res.append(terms["ds_dt"] - 0.5 * terms["beta"] * terms["grad_x"])
        else:
            res.append(std ** 3 * terms["ds_dt"] - 0.5 * eps * terms["beta"] * vp.mean_weight(t) ** 2)
    with torch.no_grad():
        return min(((r.abs().min() / r.abs().max()).item() for r in res), default=1.0)


def case_loss_sweep(model, xdim, ydim, hidden, kind, kw, batches, seed=0):
    """Fused DSM / DSM_PDE / PINN / PINN2 (the path DMIP_LOSS_PATH selects) at each batch size against the fp64 oracle:
    loss and every info entry within 3e-4 relative, every parameter gradient within 3e-3 (rms(ref) + max|ref|) — the
    tolerances of the golden-fixture and baseline-batch cases.  Returns the worst normalised error (pass: <= 1)."""
    m, params = _sweep_model(model, xdim, ydim, hidden, seed)
    worst, detail = 0.0, {}
    for B in batches:
        # a sign flip moves the gradient by about 1/B of one sample's term: keep every L1 residual 1e-4 / B of the largest
        # (>= 3e-7, above the fp32 rounding of the residuals) away from its kink
        for redraw in range(20):
            s = seed + 7919 * redraw
            prob = _sweep_problem(model, xdim, ydim, B, s)
            if _l1_margin(params, model, kind, kw, *prob) >= 1e-4 / B:
                break
        else:
            raise AssertionError("no draw keeps the L1 residuals off their kink")
        got = _sweep_library(m, model, kind, kw, *prob)
        route = "hutchinson" if kw.get("divergence_method", "exact") in ("hutchinson", "approx", "approximate") else "exact"
        key = (model, xdim, ydim, tuple(hidden), kind, tuple(sorted((k, v) for k, v in kw.items()
                                                                    if k != "divergence_method")), route, B, s)
        ref = _sweep_reference(key, params, model, kind, kw, *prob)
        e, e_loss, e_g = _sweep_errors(got, ref, 3e-4)
        detail.update({f"B{B}_loss": e_loss, f"B{B}_grad": e_g, f"B{B}_launches": float(got[3])})
        worst = max(worst, e)
    return worst, 1.0, detail


def case_loss_launches(model, xdim, ydim, hidden, kind, kw, B=37, seed=0):
    """kernel launches of one fused call under DMIP_LOSS_PATH = tc and = ffma (no reference needed)"""
    m, _ = _sweep_model(model, xdim, ydim, hidden, seed)
    prob = _sweep_problem(model, xdim, ydim, B, seed)
    counts = {}
    try:
        for path in ("tc", "ffma"):
            os.environ["DMIP_LOSS_PATH"] = path
            counts[path] = _sweep_library(m, model, kind, kw, *prob)[3]
    finally:
        os.environ.pop("DMIP_LOSS_PATH", None)
    return counts


def case_loss_rejected(model, xdim, ydim, hidden, kind, kw, match, B=37, seed=0):
    """a shape outside the documented limits must raise ValueError naming the limit and hand back no loss / gradient"""
    from dmip.models.diffusion import CDE, CDiffE
    d = xdim if model == "CDE" else xdim + ydim
    m = (CDE if model == "CDE" else CDiffE)(xdim, ydim, list(hidden))
    m.sde.to(DEV)
    prob = _sweep_problem(model, xdim, ydim, B, seed)
    assert prob[3].shape[1] == d
    try:
        _sweep_library(m, model, kind, kw, *prob)
    except ValueError as e:
        ok = match in str(e) and all(p.grad is None for p in m.sde.a.parameters())
        return (0.0 if ok else 1.0), 0.5, {"message": str(e)}
    return 1.0, 0.5, {"message": "no error"}


def _posterior_sweep_setup(xdim, hidden, ydim, seed):
    from dmip.models.diffusion import PosteriorDiffusionEstimator
    pp = make_params(seed, xdim + 1, xdim, hidden)
    lp = make_params(seed + 100, xdim + ydim + 1, xdim, hidden)
    sp = make_params(seed + 200, xdim, ydim, (256, 256, 256))
    m = PosteriorDiffusionEstimator(xdim, ydim, list(hidden))
    m.sde.a.prior_net.load_state_dict(state_dict_from_params(pp))
    m.sde.a.likelihood_net.load_state_dict(state_dict_from_params(lp))
    m.sde.to(DEV)
    # the surrogate f: R^xdim -> R^ydim in the layout of utils_scatterometry.py:9-12 (ReLU MLP, keys 0, 2, 4, 6)
    fm = torch.nn.Sequential(torch.nn.Linear(xdim, 256), torch.nn.ReLU(), torch.nn.Linear(256, 256), torch.nn.ReLU(),
                             torch.nn.Linear(256, 256), torch.nn.ReLU(), torch.nn.Linear(256, ydim))
    fm.load_state_dict({f"{i}.{n}": (W if n == "weight" else b) for i, (W, b) in zip((0, 2, 4, 6), sp)
                        for n in ("weight", "bias")})
    for p in fm.parameters():
        p.requires_grad = False
    return m, fm.to(DEV), pp, lp, sp


def _posterior_sweep_problem(xdim, ydim, B, sp, seed):
    """x ~ U[-1, 1]^xdim (the scatterometry prior box), y = f(x) + 0.01 N(0, I), t ~ U[1e-4, 1 - 1e-4], eps ~ N(0, I)"""
    g = torch.Generator().manual_seed(1000 * seed + B)
    x = torch.rand(B, xdim, generator=g) * 2 - 1
    y = (oracle.scatterometry.surrogate(sp, x) + 0.01 * torch.randn(B, ydim, generator=g)).float()
    t = torch.rand(B, 1, generator=g) * (1 - 2e-4) + 1e-4
    eps = torch.randn(B, xdim, generator=g)
    return x, y, t, eps


def _posterior_sweep_library(m, fm, lam, x, y, t, eps):
    from dmip import losses as dl
    loss_fn = dl.PosteriorLoss(fm, 0.2, 0.01, lam)
    loss, info = loss_fn(m.sde, x.to(DEV), y.to(DEV), t.to(DEV), eps.to(DEV))
    m.sde.a.zero_grad()
    loss.backward()
    grads = [p.grad.detach().cpu().double() for net in (m.sde.a.prior_net, m.sde.a.likelihood_net)
             for p in net.parameters()]
    return loss.item(), {k: v.item() for k, v in info.items()}, grads, loss_fn.last_launch_count


def case_posterior_loss_sweep(xdim, hidden, batches, ydim=23, lam=0.3, seed=0):
    """Fused PosteriorLoss (prior net, surrogate VJP at the Tweedie mean, likelihood net) at each batch size against
    ol.posterior_loss in fp64: loss and both info entries within 5e-4 relative (the tolerance of the posterior fixtures,
    case_posterior_loss: the target passes through the bf16x3 surrogate kernel), every parameter gradient of both nets
    within 3e-3 (rms(ref) + max|ref|)."""
    from oracle import losses as ol
    m, fm, pp, lp, sp = _posterior_sweep_setup(xdim, hidden, ydim, seed)
    worst, detail = 0.0, {}
    for B in batches:
        prob = _posterior_sweep_problem(xdim, ydim, B, sp, seed)
        got = _posterior_sweep_library(m, fm, lam, *prob)
        key = ("posterior", xdim, ydim, tuple(hidden), lam, B, seed)
        ref = _SWEEP_REF.get(key)
        if ref is None:
            torch.set_num_threads(max(torch.get_num_threads(), 8))
            p64 = [[(W.double().requires_grad_(True), b.double().requires_grad_(True)) for W, b in ps] for ps in (pp, lp)]
            s64 = [(W.double(), b.double()) for W, b in sp]
            loss, info = ol.posterior_loss(p64[0], p64[1], s64, *(u.double() for u in prob), lam, a=0.2, b=0.01)
            loss.backward()
            ref = (loss.item(), {k: u.item() for k, u in info.items()}, [q.grad for ps in p64 for W, b in ps for q in (W, b)])
            while len(_SWEEP_REF) >= 4:
                _SWEEP_REF.pop(next(iter(_SWEEP_REF)))
            _SWEEP_REF[key] = ref
        e, e_loss, e_g = _sweep_errors(got, ref, 5e-4)
        detail.update({f"B{B}_loss": e_loss, f"B{B}_grad": e_g, f"B{B}_launches": float(got[3])})
        worst = max(worst, e)
    return worst, 1.0, detail


def case_posterior_loss_launches(xdim, hidden, B=37, ydim=23, seed=0):
    m, fm, _, _, sp = _posterior_sweep_setup(xdim, hidden, ydim, seed)
    prob = _posterior_sweep_problem(xdim, ydim, B, sp, seed)
    counts = {}
    try:
        for path in ("tc", "ffma"):
            os.environ["DMIP_LOSS_PATH"] = path
            counts[path] = _posterior_sweep_library(m, fm, 0.3, *prob)[3]
    finally:
        os.environ.pop("DMIP_LOSS_PATH", None)
    return counts


def case_posterior_loss_rejected(xdim, hidden, match, B=37, ydim=23, seed=0):
    m, fm, _, _, sp = _posterior_sweep_setup(xdim, hidden, ydim, seed)
    prob = _posterior_sweep_problem(xdim, ydim, B, sp, seed)
    try:
        _posterior_sweep_library(m, fm, 0.3, *prob)
    except ValueError as e:
        ok = match in str(e) and all(p.grad is None for p in m.sde.a.parameters())
        return (0.0 if ok else 1.0), 0.5, {"message": str(e)}
    return 1.0, 0.5, {"message": "no error"}


# ------------------------------------------------------------------------------------------- sampler / forward sweep
# The fused samplers and the score-net forward at every kernel instantiation, state width and tile tail
# (tests/test_gpu_sampler_sweep.py; the case table and the dispatch mirror it is checked against live in
# tests/test_sampler_sweep_plan.py).  The noise is the keyed Philox stream drawn by its numpy mirror and injected, so the
# same case can also run with in-kernel Philox; particles are independent, so the fp64 oracle (oracle/ve.py, which with
# the VP-SDE and no corrector is the pinned reference sampler) integrates only the rows that are checked.
# One bound per quantity, relative to max|reference|, the bars the golden-fixture cases already meet:
SWEEP_TOL = dict(sampler=dict(fp32=2e-5, bf16=3e-3), forward=dict(fp32=2e-5, bf16=5e-3),
                 philox=dict(fp32=1e-4, bf16=2e-3), tc_vs_ffma=3e-3)
VE_SIGMA = (0.05, 4.0)          # default (sigma_min, sigma_max) of the VE-SDE cases (c['sigma']); x0 is scaled by sigma_max
_SAMPLER_REF = {}               # oracle results of the last few (case, run, rows, mutation) keys


def sweep_rows(n_obs, n_per_obs, tile, seed=0, n_random=16):
    """the rows the oracle checks: the first and last row of every `tile`-row tile of every observation (so also each
    observation's first and last row), and n_random random rows per observation"""
    rng = np.random.default_rng(seed)
    rows = set()
    for o in range(n_obs):
        base = o * n_per_obs
        for lo in range(0, n_per_obs, tile):
            rows.update((base + lo, base + min(lo + tile, n_per_obs) - 1))
        rows.update(int(r) for r in base + rng.integers(0, n_per_obs, min(n_random, n_per_obs)))
    return np.array(sorted(rows), dtype=np.int64)


def sweep_noise_key(c):
    return 7919 + c["seed"]


def sampler_problem(c, n_obs, n_per_obs):
    """make_params weights (scaled by c['gain']), observations y ~ N(0, c['y_scale']^2) (n_obs, ydim) and the keyed
    Philox draws x0 / noise / ynoise of all n_obs * n_per_obs particles"""
    variant, xdim, ydim, hidden, seed = c["variant"], c["xdim"], c["ydim"], tuple(c["hidden"]), c["seed"]
    gain = c.get("gain", 1.0)
    if variant == "DPS":
        params = make_params(seed + 100, xdim + ydim + 1, xdim, hidden, gain)
        params2 = make_params(seed, xdim + 1, xdim, hidden, gain)
    else:
        out_dim = xdim + ydim if variant == "CDiffE" else xdim
        params, params2 = make_params(seed, xdim + ydim + 1, out_dim, hidden, gain), None
    y = torch.randn(n_obs, ydim, generator=torch.Generator().manual_seed(seed)) * c.get("y_scale", 1.0)
    n_sub = c["S"] * (1 + c.get("n_corr", 0))
    gidx, key = np.arange(n_obs * n_per_obs), sweep_noise_key(c)
    normals = oracle.philox.normals
    pb = dict(params=params, params2=params2, y=y, n_obs=n_obs, n_per_obs=n_per_obs,
              x0=torch.from_numpy(normals(gidx, oracle.philox.STEP_INIT, 0, xdim, key)),
              noise=torch.from_numpy(np.stack([normals(gidx, u, 0, xdim, key) for u in range(n_sub)])), ynoise=None)
    if variant == "CDiffE":
        pb["ynoise"] = torch.from_numpy(np.stack([normals(gidx, u, 1, ydim, key) for u in range(n_sub)]))
    return pb


class _LaterSde:
    """an SDE whose coefficients are read one step late: the oracle of a kernel that takes tau from the next step"""

    def __init__(self, sde, dt):
        self.sde, self.dt, self.T, self.kind = sde, dt, sde.T, sde.kind

    def g(self, t, y):
        return self.sde.g((t - self.dt).clamp(min=0), y)

    def f(self, t, y):
        return self.sde.f((t - self.dt).clamp(min=0), y)

    def var(self, t):
        return self.sde.var((t - self.dt).clamp(min=0))

    def mean_weight(self, t):
        return self.sde.mean_weight((t - self.dt).clamp(min=0))


# kernel bugs the sweep must be able to see, stated as what the oracle computes with them (tests/test_sampler_sweep_plan.py)
SAMPLER_MUTATIONS = ("y_last_column", "neighbour_noise", "tau_next", "frozen_piece", "ynoise_previous")
FORWARD_MUTATIONS = ("input_last_column", "bias_last_output")


def sampler_oracle(c, pb, rows, mutation=None):
    """fp64 ve.pc_sampler on the given global rows, observation by observation; `mutation` injects one of
    SAMPLER_MUTATIONS: the last y column never reaches the net, the last state column takes the next row's noise, every
    step evaluates at the next step's tau, the last 8-column state piece is never updated, CDiffE re-diffuses y with the
    previous step's draws"""
    from oracle import ve
    key = (tuple(sorted((k, str(v)) for k, v in c.items())), pb["n_obs"], pb["n_per_obs"], rows.tobytes(), mutation)
    if key in _SAMPLER_REF:
        return _SAMPLER_REF[key]
    torch.set_num_threads(max(torch.get_num_threads(), 8))
    variant, xdim, S, n_corr = c["variant"], c["xdim"], c["S"], c.get("n_corr", 0)
    osde = ve.VE(*c.get("sigma", VE_SIGMA)) if c.get("sde") == "VE" else ve.VP()
    std0 = c.get("sigma", VE_SIGMA)[1] if c.get("sde") == "VE" else 1.0
    p64 = [(W.double(), b.double()) for W, b in pb["params"]]
    p2 = None if pb["params2"] is None else [(W.double(), b.double()) for W, b in pb["params2"]]
    y, x0, noise = pb["y"].double(), pb["x0"].double(), pb["noise"].double()
    ynoise = None if pb["ynoise"] is None else pb["ynoise"].double()
    net, sde = ve.net_fn(variant, p64, p2), osde
    if mutation == "y_last_column":
        y = y.clone()
        y[:, -1] = 0
        if ynoise is not None:
            ynoise = ynoise.clone()
            ynoise[:, :, -1] = 0
    elif mutation == "neighbour_noise":
        noise = noise.clone()
        noise[:, :, -1] = noise[:, :, -1].roll(-1, 1)
    elif mutation == "ynoise_previous":
        ynoise = torch.cat([ynoise[:1], ynoise[:-1]])
    elif mutation == "tau_next":
        dt = osde.T / S
        net, sde = (lambda x, cond, t, f=net: f(x, cond, (t - dt).clamp(min=0))), _LaterSde(osde, dt)
    elif mutation not in (None, "frozen_piece"):
        raise ValueError(mutation)
    rt = torch.as_tensor(rows)
    obs = rt // pb["n_per_obs"]
    out = torch.empty(len(rows), xdim, dtype=torch.float64)
    with torch.no_grad():
        for o in range(pb["n_obs"]):
            sel = obs == o
            if not bool(sel.any()):
                continue
            r = rt[sel]
            out[sel] = ve.pc_sampler(net, variant, y[o], x0[r] * std0, noise[:, r], S, sde, n_corr=n_corr, snr=0.16,
                                     ynoise=None if ynoise is None else ynoise[:, r])
    if mutation == "frozen_piece":
        lo = (xdim - 1) // 8 * 8
        out[:, lo:] = x0[rt, lo:] * std0
    while len(_SAMPLER_REF) >= 8:
        _SAMPLER_REF.pop(next(iter(_SAMPLER_REF)))
    _SAMPLER_REF[key] = out
    return out


def _sweep_sampler_model(c, pb):
    from dmip import sdes
    from dmip.models.diffusion import CDE, CDiffE, PosteriorDiffusionEstimator
    smin, smax = c.get("sigma", VE_SIGMA)
    base = sdes.VarianceExplodingSDE(sigma_min=smin, sigma_max=smax) if c.get("sde") == "VE" else None
    m = dict(CDE=CDE, CDiffE=CDiffE, DPS=PosteriorDiffusionEstimator)[c["variant"]](
        c["xdim"], c["ydim"], list(c["hidden"]), base_sde=base)
    if c["variant"] == "DPS":
        m.sde.a.prior_net.load_state_dict(state_dict_from_params(pb["params2"]))
        m.sde.a.likelihood_net.load_state_dict(state_dict_from_params(pb["params"]))
    else:
        m.sde.a.load_state_dict(state_dict_from_params(pb["params"]))
    m.sde.to(DEV)
    m.l0_split = c.get("l0_split", 4)
    return m


def _sweep_sample(m, c, pb, precision, philox=False):
    """one sampler call on all particles -> ((n_obs * n_per_obs, xdim) float64 on the host, the path that ran)"""
    kw = dict(num_samples=pb["n_per_obs"], num_steps=c["S"], precision=precision, n_corrector=c.get("n_corr", 0),
              snr=0.16, std=c.get("sigma", VE_SIGMA)[1] if c.get("sde") == "VE" else 1.0, return_tensor=True)
    if philox:
        out = m(pb["y"], seed=sweep_noise_key(c), **kw)
    else:
        inj = dict(x0=pb["x0"], noise=pb["noise"])
        if pb["ynoise"] is not None:
            inj["ynoise"] = pb["ynoise"]
        out = m(pb["y"], injected=inj, **kw)
    return out.reshape(-1, c["xdim"]).double().cpu(), m.last_precision


def case_sampler_sweep(c, paths):
    """One sampler case of the sweep at each of its runs (n_obs, n_per_obs) and precisions.  paths: precision requested
    -> the path the dispatch table says runs ('bf16' tcgen05 | 'fp32' FFMA); a call that takes another path fails.
    Every run: output finite, checked rows within SWEEP_TOL['sampler'] x max|reference of the case| of the fp64 oracle; c['philox']: the in-kernel
    Philox run within SWEEP_TOL['philox'] of the injected run.  Returns the worst err / tol (pass: <= 1)."""
    worst, detail, m = 0.0, {}, None
    runs = []
    for n_obs, n_per_obs in c["runs"]:
        pb = sampler_problem(c, n_obs, n_per_obs)
        rows = sweep_rows(n_obs, n_per_obs, 32, seed=c["seed"])
        runs.append((n_obs, n_per_obs, pb, rows, sampler_oracle(c, pb, rows)))
    # one scale per case: every run draws particle 0 of the same seeded problem, so a lone particle is measured against
    # the reference of the whole case, not against its own |x| (a single value, near 0 by chance)
    scale = max(r[4].abs().max().item() for r in runs)
    for n_obs, n_per_obs, pb, rows, ref in runs:
        m = m or _sweep_sampler_model(c, pb)
        for prec, want in paths.items():
            out, path = _sweep_sample(m, c, pb, prec)
            tag = f"{n_obs}x{n_per_obs}/{prec}"
            if path != want or not bool(torch.isfinite(out).all()):
                return float("inf"), 1.0, {tag: f"path {path} (table: {want}), finite {bool(torch.isfinite(out).all())}"}
            e = (out[rows] - ref).abs().max().item() / scale
            detail[tag] = e
            worst = max(worst, e / SWEEP_TOL["sampler"][want])
            if c.get("philox"):
                out_p, _ = _sweep_sample(m, c, pb, prec, philox=True)
                e_p = (out_p - out).abs().max().item() / out.abs().max().item()
                detail[tag + "/philox"] = e_p
                worst = max(worst, e_p / SWEEP_TOL["philox"][want])
    return worst, 1.0, detail


def persistent_particles():
    """a particle count whose 128-row tiles outnumber two rounds of the whole grid (one CTA per SM): every CTA integrates
    at least two tiles, the last round is partial, the tile count odd and the last tile partial"""
    n_sm = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    return (2 * n_sm + 3) * 128 - 50


def case_sampler_persistent(c):
    """Group B: one observation of persistent_particles() particles on the tcgen05 kernel and on the FFMA kernel, same
    injected noise: all rows within SWEEP_TOL['tc_vs_ffma'] of each other, and both within SWEEP_TOL['sampler'] of the
    fp64 oracle on the first and last row of every 128-row tile and a random sample."""
    n = persistent_particles()
    pb = sampler_problem(c, 1, n)
    m = _sweep_sampler_model(c, pb)
    rows = sweep_rows(1, n, 128, seed=c["seed"], n_random=64)
    ref = sampler_oracle(c, pb, rows)
    scale = ref.abs().max().item()
    got, worst, detail = {}, 0.0, dict(n=n)
    for prec in ("bf16", "fp32"):
        got[prec], path = _sweep_sample(m, c, pb, prec)
        if path != prec or not bool(torch.isfinite(got[prec]).all()):
            return float("inf"), 1.0, {prec: f"path {path}, finite {bool(torch.isfinite(got[prec]).all())}"}
        detail[prec] = (got[prec][rows] - ref).abs().max().item() / scale
        worst = max(worst, detail[prec] / SWEEP_TOL["sampler"][prec])
    detail["tc_vs_ffma"] = (got["bf16"] - got["fp32"]).abs().max().item() / got["fp32"].abs().max().item()
    worst = max(worst, detail["tc_vs_ffma"] / SWEEP_TOL["tc_vs_ffma"])
    return worst, 1.0, detail


def forward_problem(c, n):
    """make_params weights; x, cond, t ~ N(0, c['scale']^2) (t too: the sampler feeds the net states of about 1e2)"""
    in_dim, out_dim, hidden = c["in_dim"], c["out_dim"], tuple(c["hidden"])
    params = make_params(c["seed"], in_dim, out_dim, hidden)
    x_dim = in_dim - 1 if c["cls"] == "MLP2" else (in_dim - 1 + 1) // 2
    g = torch.Generator().manual_seed(c["seed"] + n)
    inp = torch.randn(n, in_dim, generator=g) * c["scale"]
    return params, inp[:, :x_dim], inp[:, x_dim:in_dim - 1], inp[:, in_dim - 1:]


def forward_oracle(params, x, cond, t, mutation=None):
    p64 = [(W.double(), b.double()) for W, b in params]
    t = t.double()
    if mutation == "input_last_column":
        t = torch.zeros_like(t)
    elif mutation == "bias_last_output":
        W, b = p64[-1]
        b = b.clone()
        b[-1] = 0
        p64[-1] = (W, b)
    elif mutation is not None:
        raise ValueError(mutation)
    with torch.no_grad():
        return on.mlp(p64, x.double(), cond.double(), t)


def case_forward_sweep(c, paths):
    """MLP / MLP2 forward (no autograd) at each row count of c['ns'] ('multi': persistent_particles()) and precision:
    path as the table says, output finite and within SWEEP_TOL['forward'] x max|reference of the case| of the fp64 oracle
    (all rows, or the sweep rows of the multi-round count).  Returns the worst err / tol."""
    from dmip import nets
    worst, detail = 0.0, {}
    net = None
    runs = []
    for n in c["ns"]:
        n = persistent_particles() if n == "multi" else n
        params, x, cond, t = forward_problem(c, n)
        rows = np.arange(n) if n <= 1024 else sweep_rows(1, n, 128, seed=c["seed"], n_random=64)
        runs.append((n, params, x, cond, t, rows, forward_oracle(params, x[rows], cond[rows], t[rows])))
    scale = max(r[6].abs().max().item() for r in runs)             # one scale per case, as case_sampler_sweep
    for n, params, x, cond, t, rows, ref in runs:
        if net is None:
            net = getattr(nets, c["cls"])(c["in_dim"], c["out_dim"], list(c["hidden"]), torch.nn.Tanh())
            net.load_state_dict(state_dict_from_params(params))
            net.to(DEV)
            net.l0_split = c.get("l0_split", 4)
        for prec, want in paths.items():
            net.precision = prec
            with torch.no_grad():
                if c["cls"] == "MLP2":
                    out = net(x.to(DEV), t.to(DEV))
                else:
                    out = net(x.to(DEV), cond.to(DEV), t.to(DEV))
            out = out.double().cpu()
            tag = f"n{n}/{prec}"
            if net.last_precision != want or not bool(torch.isfinite(out).all()):
                return float("inf"), 1.0, {tag: f"path {net.last_precision} (table: {want})"}
            detail[tag] = (out[rows] - ref).abs().max().item() / scale
            worst = max(worst, detail[tag] / SWEEP_TOL["forward"][want])
    return worst, 1.0, detail


def case_sampler_abi_rejects(desc, match):
    """Group H: dmip_sampler_em_vp / the C ABI refuses a descriptor outside the kernels' limits with DMIP_EINVAL and the
    message naming the limit, before anything is launched.  desc: dict of DmipSampler fields plus 'hidden' / 'hidden2'
    (widths of net / net2 after layer 0) — the weight pointers are real device buffers of those shapes."""
    _, _lib = _dmip()
    L = _lib.require_gpu()
    keep = []

    def mlp(in_dim, widths):
        m = _lib.DmipMlp()
        m.n_layers, m.in_dim, m.out_dim = len(widths), in_dim, widths[-1]
        k = in_dim
        for i, w in enumerate(widths[:_lib.MAX_LAYERS]):
            W, b = torch.zeros(w, k, device=DEV), torch.zeros(w, device=DEV)
            keep.extend((W, b))
            m.width[i], m.W[i], m.b[i] = w, W.data_ptr(), b.data_ptr()
            k = w
        return m

    d = _lib.DmipSampler()
    x, yd = desc["xdim"], desc["ydim"]
    d.variant, d.precision, d.xdim, d.ydim = desc["variant"], desc["precision"], x, yd
    d.n_obs, d.n_per_obs, d.num_steps, d.T, d.beta_min, d.beta_max, d.std = 1, 4, 2, 1.0, 0.1, 20.0, 1.0
    out_dim = x + yd if desc["variant"] == _lib.CDIFFE else x
    d.net = mlp(x + yd + 1, list(desc["hidden"]) + [out_dim])
    if desc["variant"] == _lib.DPS:
        d.net2 = mlp(x + 1, list(desc["hidden"]) + [x])
    bufs = [torch.zeros(1 << 20, device=DEV) for _ in range(3)]
    keep += bufs
    d.y, d.out, d.packed = bufs[0].data_ptr(), bufs[1].data_ptr(), bufs[2].data_ptr()
    d.packed2 = bufs[2].data_ptr() if desc["variant"] == _lib.DPS else None
    d.l0_split = 4
    ws = torch.zeros(max(L.dmip_sampler_workspace_bytes(C.byref(d)), 16), dtype=torch.uint8, device=DEV)
    keep.append(ws)
    d.workspace, d.workspace_bytes = ws.data_ptr(), ws.numel()
    rc = L.dmip_sampler_em_vp(C.byref(d), _lib.stream_ptr())
    msg = L.dmip_last_error().decode()
    torch.cuda.synchronize()
    ok = rc == -1 and match in msg and L.dmip_last_launch_count() == 0
    return (0.0 if ok else 1.0), 0.5, dict(rc=rc, message=msg)
