"""Second-order autograd through the library's score nets (pytest -m gpu).

`torch.autograd.grad(..., create_graph=True)` through MLP / MLP2.forward, then a backward through the result: the
double backward of the net runs `dmip_mlp_double_backward` (tcgen05 loss kernels, one P + T jet pass).  Checked against
fp64 torch autograd through the plain module chain, through the public API and through the reference's own literal
Score-FPE PINN loss, which must now train the net exactly as the fused PINNLoss does."""
import copy
import ctypes as C
import os
import warnings

import pytest
import torch

import gpu_cases as gc
from oracle import losses as ol, vp
from oracle.weights import make_params, state_dict_from_params

pytestmark = pytest.mark.gpu
DEV = "cuda"

# (name, x_dim, cond_dim or None for MLP2 (no cond argument) / 0 for the empty tensor, out_dim) — cat[x, cond, t]
SHAPES = [("cde_linear", 2, 2, 2), ("cdiffe_scat", 26, 0, 26), ("mlp2", 3, None, 3),
          ("in2_out1", 1, None, 1), ("in64_out64", 40, 23, 64)]
BATCHES = [1, 31, 32, 33, 65, 333]
BIG = 65536          # a P + T tile holds 32 samples, a CTA pair 64: the small batches cover partial tiles and masked CTAs


def _net(x_dim, cond_dim, out_dim, seed=0):
    from dmip import nets as dnets
    in_dim = x_dim + (cond_dim or 0) + 1
    cls = dnets.MLP2 if cond_dim is None else dnets.MLP
    net = cls(in_dim, out_dim, [512, 512, 512], torch.nn.Tanh())
    net.load_state_dict(state_dict_from_params(make_params(seed, in_dim, out_dim, (512, 512, 512))))
    return net.to(DEV)


def _call(net, x, cond, t, mlp2):
    if mlp2:
        return net(x, t)
    return net(x, cond if cond is not None else torch.Tensor([]).to(x.device).to(x.dtype), t)


def _draws(B, x_dim, cond_dim, out_dim, v_mode, seed=0):
    g = torch.Generator().manual_seed(1000 * seed + B)
    in_dim = x_dim + (cond_dim or 0) + 1
    x = torch.randn(B, x_dim, generator=g)
    cond = None if not cond_dim else torch.randn(B, cond_dim, generator=g)
    t = torch.rand(B, 1, generator=g) * 0.98 + 0.01
    u = torch.randn(B, out_dim, generator=g)
    v = torch.randn(B, in_dim, generator=g)
    if v_mode == "t_only":
        v[:, :-1] = 0.0
    return x, cond, t, u, v


def second_order(net, x, cond, t, u, v, mlp2):
    """g = grad(out, [x, cond, t], u, create_graph=True); grad((g . v).sum(), [u, x, cond, t, *params]) ->
    (first-order input gradients, second-order gradients)"""
    xx, tt, uu = (a.clone().requires_grad_(True) for a in (x, t, u))
    cc = None if cond is None else cond.clone().requires_grad_(cond.numel() > 0)
    out = _call(net, xx, cc, tt, mlp2)
    ins = [xx] + ([cc] if cc is not None and cc.numel() else []) + [tt]
    g = torch.autograd.grad(out, ins, grad_outputs=uu, create_graph=True)
    gz = torch.cat([gi.reshape(len(x), -1) for gi in g], 1)
    params = list(net.parameters())
    gg = torch.autograd.grad((gz * v).sum(), [uu] + ins + params, allow_unused=True)
    return out.detach(), [gi.detach() for gi in g], [torch.zeros_like(p) if q is None else q for q, p in
                                                     zip(gg, [uu] + ins + params)]


def _reference(net, x, cond, t, u, v, mlp2, dev):
    """fp64 torch autograd through the plain module chain"""
    ref = copy.deepcopy(net).double().to(dev)
    xr, tr, ur, vr = (a.double().to(dev) for a in (x, t, u, v))
    cr = None if cond is None else cond.double().to(dev)
    xx, tt, uu = (a.clone().requires_grad_(True) for a in (xr, tr, ur))
    cc = None if cr is None else cr.clone().requires_grad_(True)
    ins = [xx] + ([cc] if cc is not None else []) + [tt]
    out = torch.nn.Sequential.forward(ref, torch.cat([i.reshape(len(xr), -1) for i in ins], 1))
    g = torch.autograd.grad(out, ins, grad_outputs=uu, create_graph=True)
    gz = torch.cat([gi.reshape(len(xr), -1) for gi in g], 1)
    params = list(ref.parameters())
    gg = torch.autograd.grad((gz * vr).sum(), [uu] + ins + params, allow_unused=True)
    return [torch.zeros_like(p) if q is None else q for q, p in zip(gg, [uu] + ins + params)]


def _errors(got, ref, n_vec, detail=None):
    """worst normalised error: J v (entry 0) and the input gradient (entries 1 .. n_vec - 1, the columns of cat[x, cond, t]
    together) against 3e-4 of their largest |ref|, parameter gradients against 3e-3 (rms(ref) + max|ref|) — the loss
    sweep's bars for these kernels"""
    got = [a.double().cpu() for a in got]
    ref = [r.double().cpu() for r in ref]
    flat = lambda xs: torch.cat([a.reshape(a.shape[0], -1) for a in xs], 1)
    pairs = [("J v", got[0], ref[0]), ("input", flat(got[1:n_vec]), flat(ref[1:n_vec]))]
    worst = 0.0
    for i, (lab, a, r) in enumerate(pairs + [(f"param{j}", a, r) for j, (a, r) in enumerate(zip(got[n_vec:], ref[n_vec:]))]):
        if i < 2:
            e = (a - r).abs().max().item() / max(3e-4 * r.abs().max().item(), 1e-30)
        else:
            scale = r.norm().item() / max(r.numel() ** 0.5, 1.0) + r.abs().max().item()
            # the output-layer bias does not enter J: its reference gradient is 0, and the kernels' must be exactly 0
            e = (a - r).abs().max().item() / max(3e-3 * scale, 1e-30) if scale > 0 else \
                (0.0 if a.abs().max().item() == 0.0 else float("inf"))
        if detail is not None:
            detail[lab] = e
        worst = max(worst, e)
    return worst


def _check(name, x_dim, cond_dim, out_dim, B, v_mode, ref_dev="cpu"):
    net = _net(x_dim, cond_dim, out_dim)
    mlp2 = cond_dim is None
    x, cond, t, u, v = _draws(B, x_dim, cond_dim, out_dim, v_mode)
    xd, td, ud, vd = (a.to(DEV) for a in (x, t, u, v))
    cd = torch.Tensor([]).to(DEV) if cond_dim == 0 else None if cond is None else cond.to(DEV)
    _, _, got = second_order(net, xd, cd, td, ud, vd, mlp2)
    assert net.last_launch_count == 7, net.last_launch_count     # pack, P + T forward, backward, 4 weight gradients
    ref = _reference(net, x, cond, t, u, v, mlp2, ref_dev)
    n_vec = 1 + (2 if cond is None else 3)
    detail = {}
    err = _errors(got, ref, n_vec, detail)
    assert err <= 1.0, (name, B, v_mode, err, detail)


@pytest.mark.parametrize("B", BATCHES)
@pytest.mark.parametrize("name,x_dim,cond_dim,out_dim", SHAPES, ids=[s[0] for s in SHAPES])
def test_double_backward_matches_fp64_autograd(name, x_dim, cond_dim, out_dim, B):
    _check(name, x_dim, cond_dim, out_dim, B, "full")


@pytest.mark.parametrize("B", [1, 33, 333])
@pytest.mark.parametrize("name,x_dim,cond_dim,out_dim", [SHAPES[0], SHAPES[1]], ids=["cde_linear", "cdiffe_scat"])
def test_double_backward_direction_on_t_only(name, x_dim, cond_dim, out_dim, B):
    """v non-zero on the t column only: the case of ds/dt through a t leaf"""
    _check(name, x_dim, cond_dim, out_dim, B, "t_only")


@pytest.mark.parametrize("name,x_dim,cond_dim,out_dim", [SHAPES[0], SHAPES[4]], ids=["cde_linear", "in64_out64"])
def test_double_backward_large_batch(name, x_dim, cond_dim, out_dim):
    """65,536 samples (2,048 P + T tiles); the fp64 reference runs on the GPU at this size"""
    _check(name, x_dim, cond_dim, out_dim, BIG, "full", ref_dev=DEV)


# ------------------------------------------------------------------------------------------- the literal Score-FPE PINN loss
def literal_terms(net, z0, cond, t, eps, probe=None):
    """tests/test_loss_oracle_shapes.py `literal_terms` on a library net: div s from d create_graph calls (or the
    Hutchinson estimate with a probe), grad_x from a second-order call and then detached, ds/dt through a t leaf"""
    t = t.detach().clone().requires_grad_(True)
    z_t = vp.mean_weight(t) * z0 + vp.var(t) ** 0.5 * eps
    a = net(z_t, cond if cond is not None else torch.Tensor([]).to(z0.device), t)
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


def literal_pinn(net, model_kind, x, y, t, eps, ic, probe, lam, lam2, pde_metric, ic_metric):
    """PINNLoss.forward (losses.py:214-242) with the Score-FPE residual built by autograd: oracle/losses.py pinn_loss
    with the terms of `literal_terms` and the library net"""
    xdim = x.shape[1]
    z0, cond = (x, y) if model_kind == "CDE" else (torch.cat([x, y], 1), None)
    std = vp.var(t) ** 0.5
    t0 = torch.zeros_like(t)
    s0 = net(x, y, t0) / vp.beta(t0) ** 0.5
    terms = literal_terms(net, z0, cond, t, eps, probe)
    diff = s0[:, :xdim] - ic
    l_ic = lam2 * ((diff ** 2).mean(1, keepdim=True) if ic_metric == "L2" else diff.abs().mean(1, keepdim=True))
    l_dsm = ol.dsm(terms["s"], std, eps)
    l_pde = lam * ol.score_fpe(terms, pde_metric)
    loss = l_dsm.mean() + l_ic.mean() + l_pde.mean()
    return loss, {"PDE-Loss": l_pde.mean(), "Initial Condition": l_ic.mean(), "DSM-Loss": l_dsm.mean()}


PINN_CASES = [("CDE", 2, 3, "exact"), ("CDE", 4, 3, "exact"), ("CDiffE", 2, 2, "exact"), ("CDE", 4, 3, "hutchinson")]


@pytest.mark.parametrize("model,xdim,ydim,div", PINN_CASES, ids=[f"{m}_{x}+{y}_{d}" for m, x, y, d in PINN_CASES])
def test_literal_score_fpe_pinn_trains_like_the_fused_loss(model, xdim, ydim, div):
    from dmip import nets as dnets
    B = 333
    kw = dict(lam=0.5, lam2=0.7, pde_loss="FPE", ic_metric="L2", pde_metric="L2")
    if div == "hutchinson":
        kw["divergence_method"] = "hutchinson"
    m, params = gc._sweep_model(model, xdim, ydim, (512, 512, 512), 0)
    prob = gc._sweep_problem(model, xdim, ydim, B, 0)
    x, y, t, eps, ic, probe = prob
    key = ("second_order", model, xdim, ydim, div, B)
    ref = gc._sweep_reference(key, params, model, "PINN", kw, *prob)
    fused = gc._sweep_library(m, model, "PINN", kw, *prob)
    e_fused = gc._sweep_errors(fused, ref, 3e-4)[0]
    # the literal loss on the same weights and draws
    net = m.sde.a
    dnets._WARNED_EAGER[0] = False
    xd, yd, td, ed, icd, vd = (a.to(DEV) for a in prob)
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        loss, info = literal_pinn(net, model, xd, yd, td, ed, icd, vd if div == "hutchinson" else None,
                                  kw["lam"], kw["lam2"], kw["pde_metric"], kw["ic_metric"])
        net.zero_grad()
        loss.backward()
    assert not [w for w in caught if "autograd is recording" in str(w.message)], "the torch module chain ran"
    assert net.last_launch_count == 7, net.last_launch_count
    lit = (loss.item(), {k: v.item() for k, v in info.items()}, [p.grad.detach().cpu().double() for p in net.parameters()])
    e_lit = gc._sweep_errors(lit, ref, 3e-4)[0]
    assert e_fused <= 1.0 and e_lit <= 1.0, (e_fused, e_lit)


# ------------------------------------------------------------------------------------------- behaviour
def _pair(seed=0):
    net = _net(2, 2, 2, seed)
    x, cond, t, u, v = _draws(333, 2, 2, 2, "full", seed)
    return net, x.to(DEV), cond.to(DEV), t.to(DEV), u.to(DEV), v.to(DEV)


def test_first_order_results_do_not_depend_on_create_graph():
    """outputs and input gradients bitwise equal; parameter gradients (fp32 atomics in k_tcl_wgrad) within the spread of
    two create_graph=False calls"""
    net, x, cond, t, u, v = _pair()

    def run(create_graph):
        xx, cc, tt = (a.clone().requires_grad_(True) for a in (x, cond, t))
        out = net(xx, cc, tt)
        params = list(net.parameters())
        g = torch.autograd.grad(out, [xx, cc, tt] + params, grad_outputs=u, create_graph=create_graph)
        return out.detach(), [a.detach().clone() for a in g[:3]], [a.detach().clone() for a in g[3:]]

    a0, a1, a2 = run(False), run(False), run(True)
    assert torch.equal(a0[0], a2[0])
    for p, q in zip(a0[1], a2[1]):
        assert torch.equal(p, q)
    for p, q, r in zip(a0[2], a1[2], a2[2]):
        spread = (p - q).abs().max().item()
        scale = p.abs().max().item()
        assert (p - r).abs().max().item() <= max(4 * spread, 1e-6 * scale), (spread, (p - r).abs().max().item())


def test_parameter_cotangent_raises():
    net, x, cond, t, u, v = _pair()
    xx, tt = x.clone().requires_grad_(True), t.clone().requires_grad_(True)
    out = net(xx, cond, tt)
    params = list(net.parameters())
    g = torch.autograd.grad(out, [xx] + params, grad_outputs=u, create_graph=True)
    with pytest.raises(NotImplementedError, match="parameter gradient"):
        torch.autograd.grad(sum((gi ** 2).sum() for gi in g[1:]), [xx], retain_graph=True)


@pytest.mark.parametrize("cotangent", ["constant", "requires_grad"])
def test_third_order_raises(cotangent):
    """A third derivative is refused, never returned as a constant: with a constant direction v (one-hot selections, the
    divergence) the double backward's results still carry a node that raises, in autograd.grad and in a backward() of a
    loss that mixes them with first-order terms."""
    from dmip import nets as dnets
    net, x, cond, t, u, v = _pair()
    xx, tt = x.clone().requires_grad_(True), t.clone().requires_grad_(True)
    out = net(xx, cond, tt)
    g = torch.autograd.grad(out, [xx, tt], grad_outputs=u, create_graph=True)
    vv = v[:, :2].clone().requires_grad_(cotangent == "requires_grad")
    h = torch.autograd.grad((g[0] * vv).sum(), [xx], create_graph=True)[0]
    assert h.requires_grad
    # the second-order values themselves are those of a create_graph=False call
    h0 = torch.autograd.grad((g[0] * v[:, :2]).sum(), [xx], retain_graph=True)[0]
    assert torch.equal(h.detach(), h0)
    with pytest.raises(RuntimeError, match=dnets.THIRD_ORDER_MSG.split(" (")[0]):
        torch.autograd.grad(h.sum(), [xx], retain_graph=True)
    net.zero_grad()
    with pytest.raises(RuntimeError, match=dnets.THIRD_ORDER_MSG.split(" (")[0]):
        (h.sum() + out.sum()).backward()


def test_second_order_under_ffma_loss_path(monkeypatch):
    """DMIP_LOSS_PATH=ffma: every net autograd records goes through the torch module chain, twice differentiable"""
    monkeypatch.setenv("DMIP_LOSS_PATH", "ffma")
    net = _net(2, 2, 2)
    x, cond, t, u, v = _draws(65, 2, 2, 2, "full")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        _, _, got = second_order(net, x.to(DEV), cond.to(DEV), t.to(DEV), u.to(DEV), v.to(DEV), False)
    ref = _reference(net, x, cond, t, u, v, False, "cpu")
    assert _errors(got, ref, 4) <= 1.0


def test_double_backward_under_guard(monkeypatch):
    """DMIP_GUARD=1: canaries around the outputs and the workspace of dmip_mlp_double_backward"""
    monkeypatch.setenv("DMIP_GUARD", "1")
    _check("cde_linear", 2, 2, 2, 65, "full")


# ------------------------------------------------------------------------------------------- C ABI
def _desc(net, n, x, cond, t, u, v, outs):
    from dmip import _lib, nets as dnets
    keep = []
    d = dnets.DmipMlpGradGrad()
    d.net = _lib.mlp_desc(net, keep)
    d.n, d.x_dim = n, x.shape[1]
    d.cond_dim = 0 if cond is None else cond.shape[1]
    d.x, d.t, d.grad_out, d.gg_in = x.data_ptr(), t.data_ptr(), u.data_ptr(), v.data_ptr()
    d.cond = None if cond is None else cond.data_ptr()
    d.gg_out, d.grad_in, d.grad_params = (None if o is None else o.data_ptr() for o in outs)
    return d, keep


def test_abi_argument_checks():
    from dmip import nets as dnets
    L = dnets._bind_grad()
    net, x, cond, t, u, v = _pair()
    t = t.reshape(-1).contiguous()
    n = x.shape[0]
    gg = torch.empty(n, 2, device=DEV)
    gin = torch.empty(n, 5, device=DEV)
    flat = torch.empty(L.dmip_loss_grad_floats(C.byref(dnets._lib.mlp_desc(net, []))), device=DEV)
    d, keep = _desc(net, n, x, cond, t, u, v, (gg, gin, flat))
    nbytes = L.dmip_mlp_double_backward_workspace_bytes(C.byref(d))
    assert nbytes > 0
    ws = torch.empty(nbytes + 2048, dtype=torch.uint8, device=DEV)
    base = (ws.data_ptr() + 1023) & ~1023
    d.workspace, d.workspace_bytes = base, nbytes
    s = dnets._lib.stream_ptr()
    assert L.dmip_mlp_double_backward(C.byref(d), s) == 0
    torch.cuda.synchronize()
    assert L.dmip_last_launch_count() == 7
    # every output is optional: J v alone (pack + forward), J v and the input gradient (no weight gradients)
    d.grad_in, d.grad_params = None, None
    assert L.dmip_mlp_double_backward(C.byref(d), s) == 0 and L.dmip_last_launch_count() == 2
    d.grad_in = gin.data_ptr()
    assert L.dmip_mlp_double_backward(C.byref(d), s) == 0 and L.dmip_last_launch_count() == 3
    d.gg_out, d.grad_in, d.grad_params = None, None, flat.data_ptr()
    assert L.dmip_mlp_double_backward(C.byref(d), s) == 0 and L.dmip_last_launch_count() == 7
    d.gg_out, d.grad_in = gg.data_ptr(), gin.data_ptr()
    # NULL inputs
    for field in ("x", "t", "grad_out", "gg_in"):
        old = getattr(d, field)
        setattr(d, field, None)
        assert L.dmip_mlp_double_backward(C.byref(d), s) == -1, field
        setattr(d, field, old)
    old = d.cond
    d.cond = None
    assert L.dmip_mlp_double_backward(C.byref(d), s) == -1
    d.cond = old
    assert L.dmip_mlp_double_backward(None, s) == -1
    # misaligned or short workspace; a refused call leaves grad_params as it was
    flat.fill_(7.0)
    d.workspace = base + 16
    assert L.dmip_mlp_double_backward(C.byref(d), s) < 0 and b"workspace" in L.dmip_last_error()
    d.workspace, d.workspace_bytes = base, nbytes - 1
    assert L.dmip_mlp_double_backward(C.byref(d), s) < 0 and b"workspace" in L.dmip_last_error()
    d.workspace_bytes = nbytes
    old = d.gg_in
    d.gg_in = None
    assert L.dmip_mlp_double_backward(C.byref(d), s) == -1
    d.gg_in = old
    torch.cuda.synchronize()
    assert bool((flat == 7.0).all())
    # n < 0, wrong in_dim
    d.n = -1
    assert L.dmip_mlp_double_backward(C.byref(d), s) == -1
    assert L.dmip_mlp_double_backward_workspace_bytes(C.byref(d)) == 0
    d.n = n
    d.x_dim = 3
    assert L.dmip_mlp_double_backward(C.byref(d), s) == -1 and b"in_dim" in L.dmip_last_error()
    d.x_dim = 2
    # n = 0: nothing to do, the parameter gradient is zeroed
    flat.fill_(1.0)
    d.n = 0
    assert L.dmip_mlp_double_backward(C.byref(d), s) == 0
    torch.cuda.synchronize()
    assert flat.abs().max().item() == 0.0
    assert ws.numel() > 0 and keep


def test_abi_other_shapes_need_no_workspace():
    """nets outside [in <= 64] -> 512 -> 512 -> 512 -> [out <= 64]: workspace 0 (the module chain serves them)"""
    from dmip import nets as dnets
    L = dnets._bind_grad()
    net = dnets.MLP(5, 2, [256, 256, 256], torch.nn.Tanh()).to(DEV)
    x, cond, t, u, v = (a.to(DEV) for a in _draws(33, 2, 2, 2, "full"))
    d, keep = _desc(net, 33, x, cond, t.reshape(-1), u, v, (None, None, None))
    assert L.dmip_mlp_double_backward_workspace_bytes(C.byref(d)) == 0
    assert L.dmip_mlp_double_backward_workspace_bytes(None) == 0
    # and autograd through such a net is still twice differentiable (the torch chain)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        _, _, got = second_order(net, x, cond, t, u, v, False)
    assert all(torch.isfinite(g).all() for g in got)

