"""The fused score-training losses under the VE-SDE (pytest -m gpu), against the fp64 VE oracle (oracle/ve_losses.py,
pinned on the CPU by tests/test_ve_loss_oracle.py):

  sweep    DSM, DSM_PDE, PINN (Score-FPE and cScoreFPE) and PINN2 for CDE and CDiffE; d = 1 ... 4 on the forward-only
           Score-FPE route and with 'exact_adjoint' (same values), d = 5 and 31 on the adjoint route, Hutchinson; [512]^3
           nets (tcgen05) and odd widths (FFMA); batches 1, 37, 301; sigma ranges (0.01, 50) (the class default) and
           (0.05, 4); both kernel families (DMIP_LOSS_PATH), with the family that ran read from the launch counts;
  posterior PosteriorLoss at xdim 1 ... 4;
  batch    PINN at batch 65,536 against the chunked oracle;
  guard    one VE case per family with DMIP_GUARD=1 canaries;
  refusal  bad sde_kind, sigma_min <= 0, sigma_max <= sigma_min, NaN at the C ABI;
  sample_t VarianceExplodingSDE.sample_t_device (KS test against its law) and train_epoch(graph=True) on a VE model;
  trained  a VE CDE trained with train_epoch (DSM) on the linear problem, sampled with the VE sampler (bf16 and fp32),
           against the analytic linear-Gaussian posterior."""
import math
import os

import numpy as np
import pytest
import torch

import gpu_cases as gc
import test_gpu_loss_sweep as vp_sweep
from oracle import ve_losses as ove
from oracle.weights import make_params, state_dict_from_params

pytestmark = pytest.mark.gpu

DEV = "cuda"
H3 = (512, 512, 512)
BATCHES = (1, 37, 301)
SIGMAS = {"default": (0.01, 50.0), "narrow": (0.05, 4.0)}


def _loss(model, xdim, ydim, kind, kw=None, hidden=H3, batches=BATCHES):
    return dict(model=model, xdim=xdim, ydim=ydim, hidden=tuple(hidden), kind=kind, kw=dict(kw or {}), batches=batches)


PINN_FPE = vp_sweep.PINN_FPE
DSMPDE_FPE = vp_sweep.DSMPDE_FPE
PINN_CFPE = vp_sweep.PINN_CFPE
DSMPDE_CFPE = vp_sweep.DSMPDE_CFPE

CASES = {}
for _d in (1, 2, 3, 4):
    for _route in ("exact", "exact_adjoint"):
        CASES[f"cde{_d}-pinn-{_route}"] = _loss("CDE", _d, 3, "PINN", dict(PINN_FPE, divergence_method=_route))
CASES["cde2-dsmpde-exact"] = _loss("CDE", 2, 3, "DSM_PDE", DSMPDE_FPE)
CASES["cde4-dsmpde-exact_adjoint"] = _loss("CDE", 4, 3, "DSM_PDE", dict(DSMPDE_FPE, divergence_method="exact_adjoint"))
CASES["cde5-pinn-exact"] = _loss("CDE", 5, 3, "PINN", PINN_FPE)
CASES["cde31-dsmpde-exact"] = _loss("CDE", 31, 2, "DSM_PDE", DSMPDE_FPE, batches=(1, 37))
CASES["cde2-pinn-hutchinson"] = _loss("CDE", 2, 3, "PINN", dict(PINN_FPE, divergence_method="hutchinson"))
CASES["cde4-dsmpde-hutchinson"] = _loss("CDE", 4, 3, "DSM_PDE", dict(DSMPDE_FPE, divergence_method="hutchinson"))
CASES["cde2-dsm"] = _loss("CDE", 2, 3, "DSM")
CASES["cde2-pinn-cscorefpe"] = _loss("CDE", 2, 3, "PINN", PINN_CFPE)
CASES["cde2-dsmpde-cscorefpe"] = _loss("CDE", 2, 3, "DSM_PDE", DSMPDE_CFPE)
CASES["cde2-pinn2-fpe"] = _loss("CDE", 2, 3, "PINN2", dict(lam=0.5, lam2=0.7, pde_loss="FPE", ic_metric="L2"))
CASES["cde2-pinn2-cscorefpe"] = _loss("CDE", 2, 3, "PINN2", dict(lam=0.01, lam2=0.7, pde_loss="cScoreFPE", ic_metric="L1"))
CASES["cdiffe1+2-dsm"] = _loss("CDiffE", 1, 2, "DSM")
CASES["cdiffe2+2-pinn-exact"] = _loss("CDiffE", 2, 2, "PINN", PINN_FPE)
CASES["cdiffe2+3-dsmpde-exact"] = _loss("CDiffE", 2, 3, "DSM_PDE", DSMPDE_FPE)
CASES["cdiffe2+2-pinn-cscorefpe"] = _loss("CDiffE", 2, 2, "PINN", PINN_CFPE)
CASES["ffma-7x129-pinn-exact"] = _loss("CDE", 2, 3, "PINN", PINN_FPE, hidden=(7, 129))
CASES["ffma-33x1x100x7-dsm"] = _loss("CDE", 2, 3, "DSM", hidden=(33, 1, 100, 7))
CASES["ffma-128x128x127-pinn-hutchinson"] = _loss("CDE", 2, 3, "PINN", dict(PINN_FPE, divergence_method="hutchinson"),
                                                  hidden=(128, 128, 127))

_REF = {}


def _ve_model(model_kind, xdim, ydim, hidden, sigma, seed=0):
    from dmip import sdes
    from dmip.models.diffusion import CDE, CDiffE
    d = xdim if model_kind == "CDE" else xdim + ydim
    params = make_params(seed, xdim + ydim + 1, d, hidden)
    cls = CDE if model_kind == "CDE" else CDiffE
    m = cls(xdim, ydim, list(hidden), base_sde=sdes.VarianceExplodingSDE(sigma_min=sigma[0], sigma_max=sigma[1]))
    m.sde.a.load_state_dict(state_dict_from_params(params))
    m.sde.to(DEV)
    return m, params


def _is_hutch(kw):
    return kw.get("divergence_method", "exact") in ("hutchinson", "approx", "approximate")


def _ve_reference(sde, params, model_kind, kind, kw, x, y, t, eps, ic, probe):
    kw = dict(kw)
    v = probe.double() if _is_hutch(kw) else None
    kw.pop("divergence_method", None)
    p64 = [(W.double().requires_grad_(True), b.double().requires_grad_(True)) for W, b in params]
    a = [u.double() for u in (x, y, t, eps)]
    if kind == "DSM":
        loss, info = ove.dsm_loss(sde, p64, model_kind, *a), {}
    elif kind == "DSM_PDE":
        loss, info = ove.dsm_pde_loss(sde, p64, model_kind, *a, probe=v, **kw)
    else:
        fn = ove.pinn_loss if kind == "PINN" else ove.pinn2_loss
        loss, info = fn(sde, p64, model_kind, *a, ic.double(), probe=v, **kw)
    loss.backward()
    return loss.item(), {k: u.item() for k, u in info.items()}, [q.grad for W, b in p64 for q in (W, b)]


def _ve_l1_margin(sde, params, model_kind, kind, kw, x, y, t, eps, ic, probe):
    """smallest |r| / (|u| + |v|) over the entries r = u - v a loss takes the L1 norm of: how far fp32 rounding is from
    flipping the sign of r (gpu_cases._l1_margin takes |r| / max|r|, which the VE-SDE's range of scales, sigma^3 from
    1e-6 to 1.25e5 at (0.01, 50), cannot meet)"""
    p64 = [(W.double(), b.double()) for W, b in params]
    x, y, t, eps, ic = (u.double() for u in (x, y, t, eps, ic))
    pde = kw.get("pde_loss", "FPE")
    pde_metric = ("L1" if pde == "FPE" else "L2") if kind == "PINN2" else kw.get("pde_metric", "L1")
    res = []
    if kind in ("PINN", "PINN2") and kw.get("ic_metric", "L1") == "L1":
        s0 = ove.initial_score(sde, p64, x, y)[:, :x.shape[1]]
        res.append((s0 - ic, s0.abs() + ic.abs()))
    if kind != "DSM" and pde_metric == "L1":
        z0, cond, z_t, std = ove.split(sde, model_kind, x, y, t, eps)
        terms = ove.score_and_fpe_terms(sde, p64, z_t, cond, t, eps, need_space=(pde == "FPE"),
                                        probe=probe.double() if _is_hutch(kw) else None)
        if pde == "FPE":
            res.append((ove.fpe_residual(terms["ds_dt"], terms["g2"], terms["grad_x"]),
                        terms["ds_dt"].abs() + (0.5 * terms["g2"] * terms["grad_x"]).abs()))
        else:
            res.append((ove.cscore_residual(terms, eps, std),
                        (std ** 3 * terms["ds_dt"]).abs() + (0.5 * eps * terms["g2"]).abs()))
    with torch.no_grad():
        return min(((r.abs() / size.clamp_min(1e-300)).min().item() for r, size in res), default=1.0)


def _run_case(c, sigma, seed=0):
    """worst normalised error over the case's batches (pass: <= 1) and the errors per batch"""
    torch.set_num_threads(max(torch.get_num_threads(), 8))
    sde = ove.VESDE(*sigma)
    m, params = _ve_model(c["model"], c["xdim"], c["ydim"], c["hidden"], sigma, seed)
    worst, detail = 0.0, {}
    for B in c["batches"]:
        for redraw in range(20):
            s = seed + 7919 * redraw
            prob = gc._sweep_problem(c["model"], c["xdim"], c["ydim"], B, s)
            if _ve_l1_margin(sde, params, c["model"], c["kind"], c["kw"], *prob) >= 1e-4:
                break
        else:
            raise AssertionError("no draw keeps the L1 residuals off their kink")
        got = gc._sweep_library(m, c["model"], c["kind"], c["kw"], *prob)
        assert math.isfinite(got[0]), got[0]
        key = (c["model"], c["xdim"], c["ydim"], c["hidden"], c["kind"], repr(sorted(c["kw"].items())), sigma, B, s)
        if key not in _REF:
            while len(_REF) >= 4:
                _REF.pop(next(iter(_REF)))
            _REF[key] = _ve_reference(sde, params, c["model"], c["kind"], c["kw"], *prob)
        e, e_loss, e_g = gc._sweep_errors(got, _REF[key], 3e-4)
        detail.update({f"B{B}_loss": e_loss, f"B{B}_grad": e_g})
        worst = max(worst, e)
    return worst, detail


@pytest.fixture(params=["tc", "ffma"])
def loss_path(request, monkeypatch):
    monkeypatch.setenv("DMIP_LOSS_PATH", request.param)
    return request.param


@pytest.mark.parametrize("loss_path", ["tc", "ffma"], indirect=True)
@pytest.mark.parametrize("sigma", sorted(SIGMAS))
@pytest.mark.parametrize("name", sorted(CASES))
def test_ve_loss_sweep(name, sigma, loss_path):
    """loss and info means within 3e-4 relative, every parameter gradient within 3e-3 (rms(ref) + max|ref|): the
    tolerances of the VP sweep (tests/test_gpu_loss_sweep.py) for both families"""
    worst, detail = _run_case(CASES[name], SIGMAS[sigma])
    assert worst <= 1.0, (worst, detail)


@pytest.mark.parametrize("name", sorted(CASES))
def test_the_kernel_family_that_runs_is_the_one_the_table_names(name):
    """as in the VP sweep: DMIP_LOSS_PATH=ffma adds 3 launches per pass that the dispatch table puts on tcgen05"""
    c = CASES[name]
    m, _ = _ve_model(c["model"], c["xdim"], c["ydim"], c["hidden"], SIGMAS["narrow"])
    prob = gc._sweep_problem(c["model"], c["xdim"], c["ydim"], 37, 0)
    counts = {}
    try:
        for path in ("tc", "ffma"):
            os.environ["DMIP_LOSS_PATH"] = path
            counts[path] = gc._sweep_library(m, c["model"], c["kind"], c["kw"], *prob)[3]
    finally:
        os.environ.pop("DMIP_LOSS_PATH", None)
    n_tc = sum(vp_sweep.on_tcgen05(p) for p in vp_sweep.passes(c))
    assert counts["ffma"] - counts["tc"] == 3 * n_tc, (counts, n_tc)


def test_the_ve_sweep_reaches_both_families_and_both_routes():
    passes = [p for c in CASES.values() for p in vp_sweep.passes(c)]
    assert any(vp_sweep.on_tcgen05(p) for p in passes) and any(not vp_sweep.on_tcgen05(p) for p in passes)
    assert any(p[4] for p in passes) and any(p[3] for p in passes)      # grad_x pass (adjoint) and Q streams (forward)
    dims = {c["xdim"] if c["model"] == "CDE" else c["xdim"] + c["ydim"] for c in CASES.values()}
    assert {1, 2, 3, 4, 5, 31} <= dims


# --------------------------------------------------------------------------------------------- PosteriorLoss
@pytest.mark.parametrize("loss_path", ["tc", "ffma"], indirect=True)
@pytest.mark.parametrize("xdim", [1, 2, 3, 4])
def test_ve_posterior_loss(xdim, loss_path):
    """PosteriorLoss under the VE-SDE (x_t = x + sigma eps, x0_hat = x_t + sigma^2 s, alpha = 1) against the fp64 oracle:
    loss and info within 5e-4, gradients of both nets within 3e-3 (the VP posterior sweep's tolerances)"""
    from dmip import sdes
    sigma = SIGMAS["narrow"]
    sde = ove.VESDE(*sigma)
    m, fm, pp, lp, sp = gc._posterior_sweep_setup(xdim, H3, 23, 0)
    m.sde.base_sde = sdes.VarianceExplodingSDE(sigma_min=sigma[0], sigma_max=sigma[1])
    worst, detail = 0.0, {}
    for B in BATCHES:
        prob = gc._posterior_sweep_problem(xdim, 23, B, sp, 0)
        got = gc._posterior_sweep_library(m, fm, 0.3, *prob)
        torch.set_num_threads(max(torch.get_num_threads(), 8))
        p64 = [[(W.double().requires_grad_(True), b.double().requires_grad_(True)) for W, b in ps] for ps in (pp, lp)]
        s64 = [(W.double(), b.double()) for W, b in sp]
        loss, info = ove.posterior_loss(sde, p64[0], p64[1], s64, *(u.double() for u in prob), 0.3, a=0.2, b=0.01)
        loss.backward()
        ref = (loss.item(), {k: u.item() for k, u in info.items()}, [q.grad for ps in p64 for W, b in ps for q in (W, b)])
        e, e_loss, e_g = gc._sweep_errors(got, ref, 5e-4)
        detail[B] = (e_loss, e_g)
        worst = max(worst, e)
    assert worst <= 1.0, (worst, detail)


# --------------------------------------------------------------------------------------------- batch 65,536
def test_ve_pinn_at_batch_65536():
    """PINN (Score-FPE exact, L1; ic L2) on a linear CDE at batch 65,536 under the VE-SDE against the fp64 oracle in chunks
    of 4096 (sum of means): loss and info within 3e-4 relative, gradients within 3e-3 of their scale"""
    from dmip import losses as dl
    from dmip.linear_problem import LinearForwardProblem
    B, chunk = 65536, 4096
    sigma = SIGMAS["narrow"]
    sde = ove.VESDE(*sigma)
    lin = LinearForwardProblem()
    g = torch.Generator().manual_seed(7)
    x = torch.randn(B, 2, generator=g)
    y = lin(x) + 0.3 * torch.randn(B, 2, generator=g)
    t = torch.rand(B, 1, generator=g) * (1 - 2e-4) + 1e-4
    eps = torch.randn(B, 2, generator=g)
    ic = lin.score_posterior(x, y)
    m, params = _ve_model("CDE", 2, 2, H3, sigma)
    kw = dict(lam=0.001, lam2=0.1, pde_loss="FPE", ic_metric="L2", pde_metric="L1")
    icd = ic.to(DEV)
    xd, yd, td, ed = (v.to(DEV) for v in (x, y, t, eps))
    loss, info = dl.PINNLoss(lambda xx, yy: icd, **kw)(m.sde, xd, yd, xd, td, ed, None, None)
    m.sde.a.zero_grad()
    loss.backward()
    got = [p.grad.detach().cpu().double() for p in m.sde.a.parameters()]
    p64 = [(W.double().requires_grad_(True), b.double().requires_grad_(True)) for W, b in params]
    tot, tinfo = 0.0, {}
    torch.set_num_threads(max(torch.get_num_threads(), 8))
    for s in range(0, B, chunk):
        sl = slice(s, s + chunk)
        lc, ci = ove.pinn_loss(sde, p64, "CDE", *(v[sl].double() for v in (x, y, t, eps)), ic[sl].double(), **kw)
        w = (min(B, s + chunk) - s) / B
        (lc * w).backward()
        tot += lc.item() * w
        for k, v in ci.items():
            tinfo[k] = tinfo.get(k, 0.0) + v.item() * w
    e_loss = abs(loss.item() - tot) / abs(tot)
    for k, v in info.items():
        e_loss = max(e_loss, abs(v.item() - tinfo[k]) / max(abs(tinfo[k]), 1e-12))
    e_g = 0.0
    for a_, r_ in zip(got, [q.grad for W, b in p64 for q in (W, b)]):
        scale = r_.norm().item() / max(r_.numel() ** 0.5, 1.0)
        e_g = max(e_g, (a_ - r_).abs().max().item() / (3e-3 * scale + 3e-3 * r_.abs().max().item()))
    assert e_loss <= 3e-4 and e_g <= 1.0, (e_loss, e_g, loss.item(), tot)


# --------------------------------------------------------------------------------------------- guard canaries
def test_ve_losses_write_only_their_buffers():
    """DMIP_GUARD=1: canaries around the loss scalars, the flat gradient and the workspace, on both kernel families, for
    VE DSM, PINN (forward-only and adjoint Score-FPE routes, cScoreFPE) and PosteriorLoss at ragged batches"""
    from dmip import losses as dl, sdes
    os.environ["DMIP_GUARD"] = "1"
    try:
        m, _ = _ve_model("CDE", 2, 2, H3, SIGMAS["default"])
        for path in ("tc", "ffma"):
            os.environ["DMIP_LOSS_PATH"] = path
            for B in (1, 63, 65, 301):
                x, y, t = gc._dp_problem(B)
                xd, yd, td = x.to(DEV), y.to(DEV), t.to(DEV)
                e = torch.randn(B, 2, device=DEV)
                dl.dsm_fused(m, xd, yd, td, e)
                for kw in (dict(pde_loss="FPE"), dict(pde_loss="FPE", divergence_method="exact_adjoint"),
                           dict(pde_loss="cScoreFPE")):
                    fn = dl.PINNLoss(lambda xx, yy: -xx, lam=0.01, lam2=0.1, ic_metric="L2", pde_metric="L1", **kw)
                    out, _ = fn(m.sde, xd, yd, xd, td, e, None, None)
                    assert torch.isfinite(out).item()
    finally:
        os.environ.pop("DMIP_GUARD", None)
        os.environ.pop("DMIP_LOSS_PATH", None)


# --------------------------------------------------------------------------------------------- refusals at the C ABI
REFUSALS = {"kind2": (2, 0.05, 4.0, "unknown sde_kind 2"), "kind-1": (-1, 0.05, 4.0, "unknown sde_kind -1"),
            "smin0": (1, 0.0, 4.0, "0 < sigma_min < sigma_max"), "smin-neg": (1, -0.1, 4.0, "0 < sigma_min < sigma_max"),
            "smax=smin": (1, 0.5, 0.5, "0 < sigma_min < sigma_max"), "smax<smin": (1, 2.0, 1.0, "0 < sigma_min < sigma_max"),
            "nan": (1, float("nan"), 4.0, "0 < sigma_min < sigma_max"),
            "inf": (1, 0.05, float("inf"), "0 < sigma_min < sigma_max")}


@pytest.mark.parametrize("name", sorted(REFUSALS))
def test_c_abi_refuses_a_bad_sde(name, monkeypatch):
    """the library itself checks the SDE fields of DmipLoss and DmipPosteriorLoss (the Python check is bypassed here):
    DMIP_EINVAL with a message that names the limit, and no loss or gradient"""
    from dmip import _lib, losses as dl
    kind, smin, smax, match = REFUSALS[name]
    monkeypatch.setattr(_lib, "sde_params", lambda base: (kind, smin, smax))
    m, _ = _ve_model("CDE", 2, 2, H3, SIGMAS["narrow"])
    x, y, t, eps, ic, probe = gc._sweep_problem("CDE", 2, 2, 37, 0)
    with pytest.raises(ValueError, match=match):
        dl.dsm_fused(m, x.to(DEV), y.to(DEV), t.to(DEV), eps.to(DEV))
    with pytest.raises(ValueError, match=match):
        dl.PINNLoss(lambda xx, yy: -xx, **PINN_FPE)(m.sde, x.to(DEV), y.to(DEV), x.to(DEV), t.to(DEV), eps.to(DEV),
                                                      None, None)
    assert all(p.grad is None for p in m.sde.a.parameters())
    pm, fm, _, _, sp = gc._posterior_sweep_setup(2, H3, 23, 0)
    prob = gc._posterior_sweep_problem(2, 23, 37, sp, 0)
    with pytest.raises(ValueError, match=match):
        gc._posterior_sweep_library(pm, fm, 0.3, *prob)


# --------------------------------------------------------------------------------------------- t on the device, graphs
def test_ve_sample_t_device_law():
    """t = t_epsilon + u (T - t_epsilon) + eps, folded back by eps above T: a KS test against that law (2e5 draws), the
    range, and the non-debiased draw eps + u T"""
    from scipy import stats
    from dmip import sdes
    sde = sdes.VarianceExplodingSDE()
    torch.manual_seed(3)
    eps, lo, T = 1e-4, sde.t_epsilon, sde.T
    t = sde.sample_t_device([200000, 1], DEV, True, eps)
    assert t.shape == (200000, 1) and t.is_cuda and t.dtype == torch.float32
    tt = t.cpu().double().numpy().ravel()
    assert tt.min() >= lo + eps - 1e-6 and tt.max() <= T

    def cdf(v):
        v = np.asarray(v, dtype=np.float64)
        base = np.clip((v - eps - lo) / (T - lo), 0.0, 1.0)
        return base + np.clip((v - (T - eps)) / (T - lo), 0.0, None) * (v <= T)
    p = stats.kstest(tt, cdf).pvalue
    assert p > 1e-3, p
    t2 = sde.sample_t_device([100000, 1], DEV, False, eps).cpu().double().numpy().ravel()
    assert t2.min() >= eps and t2.max() <= T
    assert stats.kstest(t2[t2 < T - eps], stats.uniform(eps, T - eps).cdf).pvalue > 1e-6


def test_ve_train_epoch_captures_a_graph():
    """train_epoch(graph=True) on a VE CDE: t is drawn on the device, the step is captured, replayed, and the losses are
    finite"""
    from dmip import losses as dl, sdes
    from dmip.distributed import GraphedTrainStep
    from dmip.models.diffusion import CDE
    torch.manual_seed(0)
    X = torch.randn(4000, 2, device=DEV)
    Y = X + 0.3 * torch.randn(4000, 2, device=DEV)
    m = CDE(2, 2, [512, 512, 512], base_sde=sdes.VarianceExplodingSDE(sigma_min=0.01, sigma_max=5.0))
    opt = torch.optim.Adam(m.sde.a.parameters(), lr=1e-3)

    def loader():
        for i in range(0, 4000, 500):
            yield X[i:i + 500], Y[i:i + 500]
    for loss_fn in (dl.DSMLoss(), dl.PINNLoss(lambda xx, yy: -xx, lam=0.001, lam2=0.1, ic_metric="L2", pde_metric="L1")):
        losses = [float(m.train_epoch(opt, loss_fn, loader, graph=True)[0]) for _ in range(3)]
        assert all(np.isfinite(losses)), losses
        assert isinstance(m._graphed_step, GraphedTrainStep) and isinstance(m._graphed_step.graph, torch.cuda.CUDAGraph)


# --------------------------------------------------------------------------------------------- trained VE model
TRAIN_SIGMA = (0.01, 5.0)
# Measured on a B200 (1000 W): the trained VE CDE's 20,000 samples x 500 steps miss the posterior mean by 0.104 posterior
# std (bf16 and fp32) and the covariance by 0.073 of its largest entry; the untrained net by 2.74 std and 674.  The bars
# are >= 3x the trained errors.
TRAINED_BAR = dict(mean=0.35, cov=0.25)


def _linear_data(n=16000, seed=7):
    A = torch.tensor([[1.0, 0.5], [-0.3, 1.2]])
    b = torch.tensor([0.2, -0.1])
    sig = 0.3
    g = torch.Generator().manual_seed(seed)
    X = torch.randn(n, 2, generator=g)
    Y = X @ A.T + b + sig * torch.randn(n, 2, generator=g)
    return A, b, sig, X.to(DEV), Y.to(DEV)


def _posterior_errors(m, A, b, sig, y0, precision):
    """mean error over the posterior std and covariance error relative to |C|, for 20,000 samples of 500 steps"""
    cov = torch.linalg.inv(torch.eye(2) + A.T @ A / sig ** 2).double()
    mean = (cov @ (A.T.double() @ (y0.double() - b.double()) / sig ** 2)).numpy()
    xs = m(y0, num_samples=20000, num_steps=500, std=TRAIN_SIGMA[1], precision=precision, seed=11).astype(np.float64)
    assert np.isfinite(xs).all()
    e_mean = float(np.abs(xs.mean(0) - mean).max() / math.sqrt(cov.diagonal().max().item()))
    e_cov = float(np.abs(np.cov(xs.T) - cov.numpy()).max() / np.abs(cov.numpy()).max())
    return e_mean, e_cov


_TRAINED = {}


def _trained_ve_cde():
    if "m" not in _TRAINED:
        from dmip import losses as dl, sdes
        from dmip.models.diffusion import CDE
        torch.manual_seed(0)
        A, b, sig, X, Y = _linear_data()
        m = CDE(2, 2, [512, 512, 512], base_sde=sdes.VarianceExplodingSDE(*TRAIN_SIGMA))
        opt = torch.optim.Adam(m.sde.a.parameters(), lr=1e-3)

        def loader():
            perm = torch.randperm(X.shape[0], device=DEV)
            for i in range(0, X.shape[0], 1000):
                idx = perm[i:i + 1000]
                yield X[idx], Y[idx]
        losses = [float(m.train_epoch(opt, dl.DSMLoss(), loader)[0]) for _ in range(60)]
        assert all(np.isfinite(losses)) and losses[-1] < 0.8 * losses[0], losses
        _TRAINED["m"] = m
        _TRAINED["losses"] = losses
    return _TRAINED["m"]


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_trained_ve_cde_samples_the_linear_posterior(precision):
    """the first trained VE model: DSM through train_epoch on the linear problem, VE sampler, analytic posterior"""
    A, b, sig, _, _ = _linear_data()
    y0 = torch.tensor([0.7, -0.4])
    e_mean, e_cov = _posterior_errors(_trained_ve_cde(), A, b, sig, y0, precision)
    print(f"trained VE CDE {precision}: mean error {e_mean:.4f} std, covariance error {e_cov:.4f}, "
          f"DSM {_TRAINED['losses'][0]:.4f} -> {_TRAINED['losses'][-1]:.4f}")
    assert e_mean <= TRAINED_BAR["mean"] and e_cov <= TRAINED_BAR["cov"], (e_mean, e_cov)


def test_untrained_ve_cde_fails_the_bar():
    from dmip import sdes
    from dmip.models.diffusion import CDE
    A, b, sig, _, _ = _linear_data()
    torch.manual_seed(0)
    m = CDE(2, 2, [512, 512, 512], base_sde=sdes.VarianceExplodingSDE(*TRAIN_SIGMA))
    m.sde.to(DEV)
    e_mean, e_cov = _posterior_errors(m, A, b, sig, torch.tensor([0.7, -0.4]), "fp32")
    print(f"untrained VE CDE: mean error {e_mean:.4f} std, covariance error {e_cov:.4f}")
    assert e_mean > TRAINED_BAR["mean"] or e_cov > TRAINED_BAR["cov"], (e_mean, e_cov)
