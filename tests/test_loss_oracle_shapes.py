"""The fp64 loss oracle (oracle/losses.py) against a literal autograd statement of the Score-FPE terms, at the state
dimensions, depths and widths the fused loss kernels support but the golden fixtures do not reach (no GPU needed).

The oracle builds div s, grad_x [div s + |s|^2 + x.s] and ds/dt from forward-mode jets (explicit tangent and
second-order streams).  `tests/test_oracle_golden.py` pins that restatement to the reference's own autograd results,
but only at the fixture shapes (d in {2, 3, 26}, 3- or 4-layer nets).  Here the same terms are computed the way the
reference's ScoreFPELoss does it — one autograd call per output component, create_graph=True — and substituted into
the oracle's loss assembly; values and parameter gradients must agree to 1e-10 relative.  The GPU sweep
(tests/test_gpu_loss_sweep.py) then uses the oracle at these shapes as its reference."""
import pytest
import torch

from oracle import losses as ol, nets as onets, vp
from oracle.weights import make_params

# (model, xdim, ydim): diffused dimension d = xdim (CDE) or xdim + ydim (CDiffE).  d = 1 exists for CDE only
# (ydim >= 1); d = 4 is the largest forward-only size, d = 5 the first adjoint-route size, d = 31 the documented maximum.
SHAPES = [("CDE", 1, 2), ("CDE", 4, 3), ("CDE", 5, 2), ("CDE", 31, 2),
          ("CDiffE", 1, 3), ("CDiffE", 2, 3), ("CDiffE", 2, 29)]
# one hidden layer of width 1, an odd pair, and 8 Linear layers (DMIP_MAX_LAYERS)
HIDDEN = [(1,), (7, 129), (16,) * 7]
B = 5
TOL = 1e-10


def literal_terms(params, z0, cond, t, eps, probe=None):
    """Score-FPE terms by plain reverse-mode autograd, as ScoreFPELoss.forward forms them (losses.py:77-98):
    div s = sum_k d s_k / d x_k (create_graph=True) or, with a probe v, the Hutchinson estimate v.(d(s.v)/dx);
    grad_x = the detached gradient of div s + |s|^2 + x.s (fact Q9); ds/dt = the total derivative along x_t(t) at fixed
    eps (fact Q8), so x_t is built from a t that requires grad."""
    t = t.detach().clone().requires_grad_(True)
    z_t = vp.mean_weight(t) * z0 + vp.var(t) ** 0.5 * eps
    a = onets.mlp(params, z_t, cond, t)
    beta = vp.beta(t)
    s = a / beta ** 0.5
    n, d = s.shape
    if probe is None:
        div = sum(torch.autograd.grad(s[:, k].sum(), z_t, create_graph=True)[0][:, k] for k in range(d)).reshape(n, 1)
    else:
        jv = torch.autograd.grad((s * probe).sum(), z_t, create_graph=True)[0]
        div = (jv * probe).sum(1, keepdim=True)
    phi = div + (s ** 2).sum(1, keepdim=True) + (z_t * s).sum(1, keepdim=True)
    grad_x = torch.autograd.grad(phi.sum(), z_t, retain_graph=True)[0].detach()
    ds_dt = torch.cat([torch.autograd.grad(s[:, i].sum(), t, create_graph=True)[0] for i in range(d)], 1)
    return {"a": a, "s": s, "beta": beta, "ds_dt": ds_dt, "div_s": div, "grad_x": grad_x, "z_t": z_t}


def _literal_like_oracle(params, z_t, cond, t, z0, eps, need_space=True, probe=None):
    """drop-in for ol.score_and_fpe_terms built on `literal_terms`"""
    out = literal_terms(params, z0, cond, t, eps, probe)
    assert torch.allclose(out.pop("z_t"), z_t, rtol=1e-14, atol=1e-14)
    if not need_space:
        del out["div_s"], out["grad_x"]
    return out


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


# (oracle function, keyword arguments, uses the probe)
LOSSES = [
    ("pinn", dict(lam=0.5, lam2=0.7, pde_loss="FPE", ic_metric="L2", pde_metric="L1"), False),
    ("pinn", dict(lam=0.5, lam2=0.7, pde_loss="FPE", ic_metric="L1", pde_metric="L2"), True),
    ("pinn", dict(lam=0.5, lam2=0.7, pde_loss="cScoreFPE", ic_metric="L2", pde_metric="L1"), False),
    ("pinn2", dict(lam=0.5, lam2=0.7, pde_loss="FPE", ic_metric="L2"), False),
    ("pinn2", dict(lam=0.5, lam2=0.7, pde_loss="cScoreFPE", ic_metric="L1"), False),
    ("dsm_pde", dict(lam=0.3, pde_loss="FPE", pde_metric="L2"), False),
    ("dsm_pde", dict(lam=0.3, pde_loss="FPE", pde_metric="L1"), True),
]


def _run(fn, params, model, x, y, t, eps, ic, probe, kw):
    p = [(W.clone().requires_grad_(True), b.clone().requires_grad_(True)) for W, b in params]
    if fn == "dsm_pde":
        loss, info = ol.dsm_pde_loss(p, model, x, y, t, eps, probe=probe, **kw)
    else:
        loss, info = getattr(ol, fn + "_loss")(p, model, x, y, t, eps, ic, probe=probe, **kw)
    loss.backward()
    return loss.detach(), {k: v.detach() for k, v in info.items()}, [q.grad for pair in p for q in pair]


@pytest.mark.parametrize("hidden", HIDDEN, ids=lambda h: "x".join(map(str, h)) if len(set(h)) > 1 else f"{h[0]}x{len(h)}")
@pytest.mark.parametrize("model,xdim,ydim", SHAPES, ids=lambda v: str(v))
def test_score_fpe_terms_match_literal_autograd(model, xdim, ydim, hidden):
    params, x, y, t, eps, ic, probe = _problem(model, xdim, ydim, hidden)
    z0, cond, z_t, _ = ol._split(model, x, y, t, eps)
    for v in (None, probe):
        ref = ol.score_and_fpe_terms(params, z_t, cond, t, z0, eps, probe=v)
        lit = literal_terms(params, z0, cond, t, eps, v)
        for k in ("s", "ds_dt", "div_s", "grad_x"):
            assert ref[k].shape == lit[k].shape, k
            err = _rel(ref[k], lit[k])
            assert err <= TOL, (k, "hutchinson" if v is not None else "exact", err)


@pytest.mark.parametrize("hidden", HIDDEN, ids=lambda h: "x".join(map(str, h)) if len(set(h)) > 1 else f"{h[0]}x{len(h)}")
@pytest.mark.parametrize("model,xdim,ydim", SHAPES, ids=lambda v: str(v))
def test_losses_and_gradients_match_literal_autograd(model, xdim, ydim, hidden, monkeypatch):
    """the oracle's PINN / PINN2 / DSM_PDE losses, info entries and parameter gradients, with the jet terms replaced by
    the literal autograd ones (the loss assembly around them is the part the golden fixtures pin)"""
    params, x, y, t, eps, ic, probe = _problem(model, xdim, ydim, hidden)
    for fn, kw, hutch in LOSSES:
        v = probe if hutch else None
        ref = _run(fn, params, model, x, y, t, eps, ic, v, kw)
        with monkeypatch.context() as mp:
            mp.setattr(ol, "score_and_fpe_terms", _literal_like_oracle)
            lit = _run(fn, params, model, x, y, t, eps, ic, v, kw)
        what = (fn, kw, "hutchinson" if hutch else "exact")
        assert abs(lit[0] - ref[0]).item() <= TOL * abs(ref[0]).item(), (what, lit[0].item(), ref[0].item())
        for k in ref[1]:
            assert abs(lit[1][k] - ref[1][k]).item() <= TOL * abs(ref[1][k]).item(), (what, k)
        for i, (g_lit, g_ref) in enumerate(zip(lit[2], ref[2])):
            err = _rel(g_lit, g_ref)
            assert err <= TOL, (what, "parameter", i, err)
