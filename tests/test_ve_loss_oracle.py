"""The VE-SDE loss oracle (oracle/ve_losses.py) pinned on the CPU, before any kernel is compared with it:

  1. its jet Score-FPE terms and its losses against a literal autograd statement (one autograd.grad per component,
     create_graph=True, as tests/test_loss_oracle_shapes.py does for the VP oracle): values and parameter gradients 1e-10;
  2. the PDE itself, with exact scores in place of the net: for data x0 ~ sum_k w_k N(m_k, C_k) the perturbed density is
     p_t = sum_k w_k N(m_k, C_k + sigma(t)^2 I), and its score must make the VE Score-FPE residual vanish; the conditional
     score -eps / sigma must make the cScoreFPE residual vanish.  The same harness with the VP density and the VP residual
     vanishes too, and drops out of balance when the x.s term is removed: the harness tells the two SDEs apart;
  3. the one mapping from a model's base_sde to the kernels' (sde_kind, p0, p1), and its refusals."""
import math

import pytest
import torch

from oracle import losses as ol, nets as onets, ve_losses as ove, vp
from oracle.weights import make_params

SHAPES = [("CDE", 1, 2), ("CDE", 2, 3), ("CDE", 4, 3), ("CDE", 5, 2), ("CDE", 31, 2), ("CDiffE", 2, 3)]
HIDDEN = [(1,), (7, 129), (16,) * 7]          # 2, 3 and 8 Linear layers
SIGMAS = [(0.01, 50.0), (0.05, 4.0)]
B = 5
TOL = 1e-10


def literal_terms(sde, params, z0, cond, t, eps, probe=None):
    """Score-FPE terms of the VE-SDE by plain reverse-mode autograd: x_t = z0 + sigma(t) eps with t requiring grad (the
    total derivative along x_t(t), fact Q8), s = a / g, div s per component (or v.(d(s.v)/dx)), grad_x of
    div s + |s|^2 detached (fact Q9; no x.s term: f = 0)."""
    t = t.detach().clone().requires_grad_(True)
    z_t = z0 + sde.sigma(t) * eps
    a = onets.mlp(params, z_t, cond, t)
    g2 = sde.g2(t)
    s = a / g2 ** 0.5
    n, d = s.shape
    if probe is None:
        div = sum(torch.autograd.grad(s[:, k].sum(), z_t, create_graph=True)[0][:, k] for k in range(d)).reshape(n, 1)
    else:
        jv = torch.autograd.grad((s * probe).sum(), z_t, create_graph=True)[0]
        div = (jv * probe).sum(1, keepdim=True)
    phi = div + (s ** 2).sum(1, keepdim=True)
    grad_x = torch.autograd.grad(phi.sum(), z_t, retain_graph=True)[0].detach()
    ds_dt = torch.cat([torch.autograd.grad(s[:, i].sum(), t, create_graph=True)[0] for i in range(d)], 1)
    return {"a": a, "s": s, "g2": g2, "ds_dt": ds_dt, "div_s": div, "grad_x": grad_x, "z_t": z_t}


def _problem(model, xdim, ydim, hidden, seed=0):
    d = xdim if model == "CDE" else xdim + ydim
    params = [(W.double(), b.double()) for W, b in make_params(seed, xdim + ydim + 1, d, hidden)]
    g = torch.Generator().manual_seed(seed + 1)
    x = torch.randn(B, xdim, generator=g, dtype=torch.float64)
    y = torch.randn(B, ydim, generator=g, dtype=torch.float64)
    t = torch.rand(B, 1, generator=g, dtype=torch.float64) * (1 - 2e-4) + 1e-4
    eps = torch.randn(B, d, generator=g, dtype=torch.float64)
    ic = torch.randn(B, xdim, generator=g, dtype=torch.float64)
    probe = torch.randint(0, 2, (B, d), generator=g).double() * 2 - 1
    return params, x, y, t, eps, ic, probe


def _rel(got, ref):
    return ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-300)).item()


def _hid(h):
    return "x".join(map(str, h)) if len(set(h)) > 1 else f"{h[0]}x{len(h)}"


# --------------------------------------------------------------------------------------------- 1. literal autograd
@pytest.mark.parametrize("sigma", SIGMAS, ids=lambda s: f"{s[0]}-{s[1]}")
@pytest.mark.parametrize("hidden", HIDDEN, ids=_hid)
@pytest.mark.parametrize("model,xdim,ydim", SHAPES, ids=lambda v: str(v))
def test_ve_score_fpe_terms_match_literal_autograd(model, xdim, ydim, hidden, sigma):
    sde = ove.VESDE(*sigma)
    params, x, y, t, eps, ic, probe = _problem(model, xdim, ydim, hidden)
    z0, cond, z_t, _ = ove.split(sde, model, x, y, t, eps)
    for v in (None, probe):
        ref = ove.score_and_fpe_terms(sde, params, z_t, cond, t, eps, probe=v)
        lit = literal_terms(sde, params, z0, cond, t, eps, v)
        assert torch.allclose(lit["z_t"], z_t, rtol=1e-14, atol=1e-14)
        for k in ("s", "ds_dt", "div_s", "grad_x"):
            assert ref[k].shape == lit[k].shape, k
            err = _rel(ref[k], lit[k])
            assert err <= TOL, (k, "hutchinson" if v is not None else "exact", err)


LOSSES = [
    ("pinn", dict(lam=0.5, lam2=0.7, pde_loss="FPE", ic_metric="L2", pde_metric="L1"), False),
    ("pinn", dict(lam=0.5, lam2=0.7, pde_loss="FPE", ic_metric="L1", pde_metric="L2"), True),
    ("pinn", dict(lam=0.5, lam2=0.7, pde_loss="cScoreFPE", ic_metric="L2", pde_metric="L1"), False),
    ("pinn2", dict(lam=0.5, lam2=0.7, pde_loss="FPE", ic_metric="L2"), False),
    ("pinn2", dict(lam=0.5, lam2=0.7, pde_loss="cScoreFPE", ic_metric="L1"), False),
    ("dsm_pde", dict(lam=0.3, pde_loss="FPE", pde_metric="L2"), False),
    ("dsm_pde", dict(lam=0.3, pde_loss="FPE", pde_metric="L1"), True),
    ("dsm_pde", dict(lam=0.3, pde_loss="cScoreFPE", pde_metric="L2"), False),
]


def _run(sde, fn, params, model, x, y, t, eps, ic, probe, kw):
    p = [(W.clone().requires_grad_(True), b.clone().requires_grad_(True)) for W, b in params]
    if fn == "dsm_pde":
        loss, info = ove.dsm_pde_loss(sde, p, model, x, y, t, eps, probe=probe, **kw)
    else:
        loss, info = getattr(ove, fn + "_loss")(sde, p, model, x, y, t, eps, ic, probe=probe, **kw)
    loss.backward()
    return loss.detach(), {k: v.detach() for k, v in info.items()}, [q.grad for pair in p for q in pair]


def _literal_like_oracle(sde, params, z_t, cond, t, eps, need_space=True, probe=None):
    """drop-in for ove.score_and_fpe_terms built on `literal_terms`"""
    z0 = z_t - sde.sigma(t) * eps
    out = literal_terms(sde, params, z0, cond, t, eps, probe)
    out.pop("z_t")
    if not need_space:
        del out["div_s"], out["grad_x"]
    return out


@pytest.mark.parametrize("hidden", HIDDEN, ids=_hid)
@pytest.mark.parametrize("model,xdim,ydim", SHAPES, ids=lambda v: str(v))
def test_ve_losses_and_gradients_match_literal_autograd(model, xdim, ydim, hidden, monkeypatch):
    """PINN / PINN2 / DSM_PDE under the VE-SDE with the jet terms replaced by the literal autograd ones: loss, info
    entries and parameter gradients; and DSM against its direct autograd statement"""
    sde = ove.VESDE(0.05, 4.0)
    params, x, y, t, eps, ic, probe = _problem(model, xdim, ydim, hidden)
    for fn, kw, hutch in LOSSES:
        v = probe if hutch else None
        ref = _run(sde, fn, params, model, x, y, t, eps, ic, v, kw)
        with monkeypatch.context() as mp:
            mp.setattr(ove, "score_and_fpe_terms", _literal_like_oracle)
            lit = _run(sde, fn, params, model, x, y, t, eps, ic, v, kw)
        what = (fn, kw, "hutchinson" if hutch else "exact")
        assert abs(lit[0] - ref[0]).item() <= TOL * abs(ref[0]).item(), (what, lit[0].item(), ref[0].item())
        for k in ref[1]:
            assert abs(lit[1][k] - ref[1][k]).item() <= TOL * abs(ref[1][k]).item(), (what, k)
        for i, (g_lit, g_ref) in enumerate(zip(lit[2], ref[2])):
            assert _rel(g_lit, g_ref) <= TOL, (what, "parameter", i)
    # DSM: 1/2 sum (s sigma + eps)^2 with s = a(x + sigma eps, y, t) / (sigma sqrt(2 lr))
    z0 = x if model == "CDE" else torch.cat([x, y], 1)
    cond = y if model == "CDE" else None
    sig = sde.smin * (sde.smax / sde.smin) ** t
    a = onets.mlp(params, z0 + sig * eps, cond, t)
    want = (((a / (sig * math.sqrt(2 * math.log(sde.smax / sde.smin))) * sig + eps) ** 2).sum(1) / 2).mean()
    assert abs(ove.dsm_loss(sde, params, model, x, y, t, eps) - want).item() <= TOL * want.item()


def test_ve_initial_condition_divides_by_g0():
    sde = ove.VESDE(0.05, 4.0)
    params, x, y, *_ = _problem("CDE", 2, 3, (7, 129))
    a0 = onets.mlp(params, x, y, torch.zeros(B, 1, dtype=torch.float64))
    g0 = 0.05 * math.sqrt(2 * math.log(4.0 / 0.05))
    assert _rel(ove.initial_score(sde, params, x, y), a0 / g0) <= 1e-14


# --------------------------------------------------------------------------------------------- 2. the PDE itself
def _mixture(d, seed):
    """two Gaussian components N(m_k, C_k) in d dimensions, weights 0.3 / 0.7"""
    g = torch.Generator().manual_seed(seed)
    comps = []
    for _ in range(2):
        A = torch.randn(d, d, generator=g, dtype=torch.float64) * 0.5
        comps.append((torch.randn(d, generator=g, dtype=torch.float64), A @ A.T + 0.3 * torch.eye(d, dtype=torch.float64)))
    return [0.3, 0.7], comps


def _log_p(x, t, weights, comps, mean_w, var):
    """log of sum_k w_k N(x; mean_w(t) m_k, mean_w(t)^2 C_k + var(t) I), x (B, d), t (B, 1)"""
    d = x.shape[1]
    eye = torch.eye(d, dtype=x.dtype)
    terms = []
    for w, (m, Cm) in zip(weights, comps):
        al, v = mean_w(t), var(t)                                   # (B, 1)
        S = al[:, :, None] ** 2 * Cm + v[:, :, None] * eye          # (B, d, d)
        r = x - al * m
        sol = torch.linalg.solve(S, r.unsqueeze(-1)).squeeze(-1)
        terms.append(math.log(w) - 0.5 * (r * sol).sum(1) - 0.5 * torch.logdet(S) - 0.5 * d * math.log(2 * math.pi))
    return torch.logsumexp(torch.stack(terms, 1), 1)


def _exact_score_jets(x, t, weights, comps, mean_w, var, g2):
    """a = g s of the exact score s = grad log p_t, its partial time derivative a_t (x fixed), J = da/dx and
    gtr[k] = sum_i d^2 a_i / dx_i dx_k — the quantities the loss kernels take from the net's jets"""
    x = x.detach().clone().requires_grad_(True)
    t = t.detach().clone().requires_grad_(True)
    lp = _log_p(x, t, weights, comps, mean_w, var)
    s = torch.autograd.grad(lp.sum(), x, create_graph=True)[0]
    a = g2(t) ** 0.5 * s
    n, d = a.shape
    a_t = torch.cat([torch.autograd.grad(a[:, i].sum(), t, create_graph=True)[0] for i in range(d)], 1)
    J = torch.stack([torch.autograd.grad(a[:, i].sum(), x, create_graph=True)[0] for i in range(d)], 1)   # [b, i, k]
    tr = torch.diagonal(J, dim1=1, dim2=2).sum(1)
    gtr = torch.autograd.grad(tr.sum(), x, retain_graph=True)[0]
    return x.detach(), t.detach(), a.detach(), a_t.detach(), J.detach(), gtr.detach()


def _points(d, seed=3, n=64):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(n, d, generator=g, dtype=torch.float64) * 2,
            torch.rand(n, 1, generator=g, dtype=torch.float64) * 0.98 + 0.01)


@pytest.mark.parametrize("sigma", SIGMAS, ids=lambda s: f"{s[0]}-{s[1]}")
@pytest.mark.parametrize("d", [1, 2, 4])
def test_exact_ve_score_solves_the_ve_score_fpe(d, sigma):
    """R = ds/dt - g^2/2 grad_x [div s + |s|^2] = 0 for the exact score of the VE-perturbed data, with ds/dt and
    grad_x formed exactly as the oracle forms them from a, a_t, J, gtr (ove.ds_dt, ove.grad_phi, ove.fpe_residual)"""
    sde = ove.VESDE(*sigma)
    weights, comps = _mixture(d, seed=d)
    x, t = _points(d)
    x, t, a, a_t, J, gtr = _exact_score_jets(x, t, weights, comps, lambda t: torch.ones_like(t),
                                             lambda t: sde.sigma(t) ** 2, sde.g2)
    R = ove.fpe_residual(ove.ds_dt(sde, a, a_t, t), sde.g2(t), ove.grad_phi(a, J, gtr, sde.g2(t)))
    scale = ove.ds_dt(sde, a, a_t, t).abs().max()
    assert scale > 1e-3
    assert (R.abs().max() / scale).item() <= 1e-10


def _vp_grad_phi(a, J, gtr, x, g2, with_xs=True):
    """the VP row of the table: gtr / g + 2 J^T a / g^2 + (a + J^T x) / g  (the last term is grad_x (x.s))"""
    g = g2 ** 0.5
    out = gtr / g + 2 * torch.einsum("bik,bi->bk", J, a) / g2
    if with_xs:
        out = out + (a + torch.einsum("bik,bi->bk", J, x)) / g
    return out


@pytest.mark.parametrize("d", [1, 2, 4])
def test_the_harness_tells_vp_from_ve(d):
    """the same harness with the VP-perturbed density and the VP residual (ds/dt = a_t / g - a beta' / (2 beta g),
    phi with the x.s term) vanishes; without the x.s term it does not, nor does the VE residual on the VP density"""
    weights, comps = _mixture(d, seed=10 + d)
    x, t = _points(d, seed=11)
    x, t, a, a_t, J, gtr = _exact_score_jets(x, t, weights, comps, vp.mean_weight, vp.var, vp.beta)
    b = vp.beta(t)
    ds = a_t / b ** 0.5 - a * (vp.BETA_MAX - vp.BETA_MIN) / (2 * b ** 1.5)
    scale = ds.abs().max()
    R = ds - 0.5 * b * _vp_grad_phi(a, J, gtr, x, b)
    assert (R.abs().max() / scale).item() <= 1e-10
    R_no_xs = ds - 0.5 * b * _vp_grad_phi(a, J, gtr, x, b, with_xs=False)
    assert (R_no_xs.abs().max() / scale).item() > 1e-2
    # the oracle's VP loss formula (oracle/losses.py score_fpe) agrees with the table's VP row here
    R_oracle = ds - 0.5 * b * _vp_grad_phi(a, J, gtr, x, b)
    terms = {"ds_dt": ds, "beta": b, "grad_x": _vp_grad_phi(a, J, gtr, x, b)}
    assert (ol.score_fpe(terms, "L1") - R_oracle.abs().mean(1, keepdim=True)).abs().max().item() <= 1e-12 * scale.item()
    # and the VE residual on a VE density does not vanish when the VP formula is used on it
    sde = ove.VESDE(0.05, 4.0)
    x, t, a, a_t, J, gtr = _exact_score_jets(x, t, weights, comps, lambda t: torch.ones_like(t),
                                             lambda t: sde.sigma(t) ** 2, sde.g2)
    ds = ove.ds_dt(sde, a, a_t, t)
    wrong = ds - 0.5 * sde.g2(t) * _vp_grad_phi(a, J, gtr, x, sde.g2(t))
    assert (wrong.abs().max() / ds.abs().max()).item() > 1e-2


@pytest.mark.parametrize("sigma", SIGMAS, ids=lambda s: f"{s[0]}-{s[1]}")
def test_conditional_score_solves_the_ve_cscore_fpe(sigma):
    """s = -eps / sigma(t) along x_t = z0 + sigma eps: std^3 ds/dt - eps g^2 / 2 = 0 (ove.cscore_residual); and the VP
    conditional score -eps / std against the VP cScoreFPE of oracle/losses.py"""
    sde = ove.VESDE(*sigma)
    g = torch.Generator().manual_seed(4)
    eps = torch.randn(32, 3, generator=g, dtype=torch.float64)
    t = (torch.rand(32, 1, generator=g, dtype=torch.float64) * 0.98 + 0.01).requires_grad_(True)
    s = -eps / sde.sigma(t)
    ds = torch.cat([torch.autograd.grad(s[:, i].sum(), t, retain_graph=True)[0] for i in range(3)], 1)
    r = ove.cscore_residual({"ds_dt": ds, "g2": sde.g2(t)}, eps, sde.sigma(t))
    assert (r.abs().max() / (sde.sigma(t) ** 3 * ds).abs().max()).item() <= 1e-12
    std = vp.var(t) ** 0.5
    s = -eps / std
    ds = torch.cat([torch.autograd.grad(s[:, i].sum(), t, retain_graph=True)[0] for i in range(3)], 1)
    loss = ol.cscore_fpe({"ds_dt": ds, "beta": vp.beta(t)}, t, eps, std, "L1")
    assert (loss.max() / (std ** 3 * ds).abs().sum(1).max()).item() <= 1e-12
    # the VP formula on the VE conditional score does not vanish
    s = -eps / sde.sigma(t)
    ds = torch.cat([torch.autograd.grad(s[:, i].sum(), t, retain_graph=True)[0] for i in range(3)], 1)
    wrong = sde.sigma(t) ** 3 * ds - 0.5 * eps * vp.beta(t) * vp.mean_weight(t) ** 2
    assert (wrong.abs().max() / (sde.sigma(t) ** 3 * ds).abs().max()).item() > 1e-2


def test_ve_xdot_is_the_time_derivative_of_x_t():
    sde = ove.VESDE(0.05, 4.0)
    t = torch.tensor([[0.3], [0.8]], dtype=torch.float64, requires_grad=True)
    eps = torch.tensor([[0.5, -1.0], [2.0, 0.1]], dtype=torch.float64)
    z0 = torch.tensor([[1.0, 2.0], [-1.0, 0.0]], dtype=torch.float64)
    x_t, _ = sde.perturb(t, z0, eps)
    dx = torch.cat([torch.autograd.grad(x_t[:, i].sum(), t, retain_graph=True)[0] for i in range(2)], 1)
    assert _rel(sde.xdot(t, eps), dx) <= 1e-14


# --------------------------------------------------------------------------------------------- 3. the SDE mapping
def test_sde_params_maps_each_base_sde():
    from dmip import _lib, sdes
    assert _lib.sde_params(sdes.VariancePreservingSDE()) == (_lib.SDE_VP, 0.1, 20.0)
    assert _lib.sde_params(sdes.VariancePreservingSDE(beta_min=0.2, beta_max=10.0)) == (_lib.SDE_VP, 0.2, 10.0)
    assert _lib.sde_params(sdes.VarianceExplodingSDE()) == (_lib.SDE_VE, 0.01, 50.0)
    assert _lib.sde_params(sdes.VarianceExplodingSDE(sigma_min=0.05, sigma_max=4.0)) == (_lib.SDE_VE, 0.05, 4.0)


def test_set_sde_fills_the_descriptors():
    from dmip import _lib, losses, posterior, sdes
    for cls in (_lib.DmipSampler, losses.DmipLoss, posterior.DmipPosteriorLoss):
        d = cls()
        _lib.set_sde(d, sdes.VarianceExplodingSDE(sigma_min=0.05, sigma_max=4.0))
        assert (d.sde_kind, d.beta_min, d.beta_max) == (_lib.SDE_VE, 0.0, 0.0)
        assert (d.sigma_min, d.sigma_max) == pytest.approx((0.05, 4.0))
        d = cls()
        _lib.set_sde(d, sdes.VariancePreservingSDE())
        assert (d.sde_kind, d.sigma_min, d.sigma_max) == (_lib.SDE_VP, 0.0, 0.0)
        assert (d.beta_min, d.beta_max) == pytest.approx((0.1, 20.0))


@pytest.mark.parametrize("smin,smax", [(0.0, 1.0), (-0.1, 1.0), (1.0, 1.0), (2.0, 1.0), (float("nan"), 1.0),
                                       (0.1, float("inf"))])
def test_sde_params_refuses_a_bad_ve_range(smin, smax):
    from dmip import _lib, sdes
    with pytest.raises(ValueError, match="VE-SDE needs finite 0 < sigma_min < sigma_max"):
        _lib.sde_params(sdes.VarianceExplodingSDE(sigma_min=smin, sigma_max=smax))


def test_sde_params_refuses_an_unknown_sde():
    from dmip import _lib
    with pytest.raises(ValueError, match="VP-SDE .* or sdes.VarianceExplodingSDE"):
        _lib.sde_params(object())


def test_ve_sample_t_host_law():
    """the host draw the device draw restates: uniform on [t_epsilon, T] + eps, folded back below T"""
    from dmip import sdes
    sde = sdes.VarianceExplodingSDE()
    torch.manual_seed(0)
    t = sde.sample_debiasing_t([20000, 1])
    assert t.min().item() >= sde.t_epsilon and t.max().item() <= sde.T
