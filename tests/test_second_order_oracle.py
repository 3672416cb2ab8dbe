"""The decomposition behind dmip_mlp_double_backward, checked in float64 on the CPU (no GPU needed).

The backward of the score net maps (z = cat[x, cond, t], params, u) to (J^T u, d(u^T a)/d params), J = da/dz.  Its
backward with a cotangent v on J^T u is the gradient of <v, J^T u> = u^T J v, and J v is the tangent stream T of the
forward-mode jets with input direction v.  So d/du = J v, and the gradients w.r.t. z and the parameters are a reverse
pass through the P + T jets with output adjoints P: 0 and T: u — what the tcgen05 loss kernels compute for post = 5.
Here that statement, through `oracle.nets.mlp_jets`, must equal torch's own double backward through `oracle.nets.mlp`."""
import pytest
import torch

from oracle import nets as onets
from oracle.weights import make_params

TOL = 1e-10
B = 6

# (name, x_dim, cond_dim or None for no cond argument (MLP2) / 0 for the empty tensor, out_dim)
SHAPES = [("cde_linear", 2, 2, 2), ("cdiffe_scat", 26, 0, 26), ("mlp2", 3, None, 3),
          ("in2_out1", 1, None, 1), ("in64_out64", 40, 23, 64)]


def _problem(x_dim, cond_dim, out_dim, seed=0):
    in_dim = x_dim + (cond_dim or 0) + 1
    params = [(W.double(), b.double()) for W, b in make_params(seed, in_dim, out_dim, (512, 512, 512))]
    g = torch.Generator().manual_seed(seed + 1)
    x = torch.randn(B, x_dim, generator=g, dtype=torch.float64)
    cond = None if cond_dim is None else torch.randn(B, cond_dim, generator=g, dtype=torch.float64)
    t = torch.rand(B, generator=g, dtype=torch.float64) * 0.98 + 0.01
    u = torch.randn(B, out_dim, generator=g, dtype=torch.float64)
    v = torch.randn(B, in_dim, generator=g, dtype=torch.float64)
    return params, x, cond, t, u, v


def _leaves(params, x, cond, t, u):
    p = [(W.clone().requires_grad_(True), b.clone().requires_grad_(True)) for W, b in params]
    xs = [x.clone().requires_grad_(True), None if cond is None else cond.clone().requires_grad_(True),
          t.clone().requires_grad_(True), u.clone().requires_grad_(True)]
    return p, xs


def torch_double_backward(params, x, cond, t, u, v):
    """grad(a, [x, cond, t], grad_outputs=u, create_graph=True), then grad((g . v).sum(), [u, x, cond, t, params])"""
    p, (xx, cc, tt, uu) = _leaves(params, x, cond, t, u)
    a = onets.mlp(p, xx, cc if cc is not None else torch.Tensor([]).double(), tt)
    ins = [xx] + ([cc] if cc is not None and cc.numel() else []) + [tt]
    g = torch.autograd.grad(a, ins, grad_outputs=uu, create_graph=True)
    gz = torch.cat([gi.reshape(len(x), -1) for gi in g], 1)
    flat = [q for pair in p for q in pair]
    wrt = [uu] + ins + flat
    return torch.autograd.grad((gz * v).sum(), wrt, allow_unused=True)


def jet_double_backward(params, x, cond, t, u, v):
    """J v from the T stream; the rest from a reverse pass through the P + T jets seeded with abar_P = 0, abar_T = u"""
    p, (xx, cc, tt, _) = _leaves(params, x, cond, t, u)
    ins = [xx] + ([cc] if cc is not None and cc.numel() else []) + [tt]
    z = torch.cat([xx] + ([cc] if cc is not None and cc.numel() else []) + [tt.reshape(-1, 1)], 1)
    out_p, (out_t,), _ = onets.mlp_jets(p, z, [v])
    flat = [q for pair in p for q in pair]
    grads = torch.autograd.grad([out_p, out_t], ins + flat, grad_outputs=[torch.zeros_like(out_p), u],
                                allow_unused=True)
    return (out_t.detach(),) + grads


@pytest.mark.parametrize("name,x_dim,cond_dim,out_dim", SHAPES, ids=[s[0] for s in SHAPES])
@pytest.mark.parametrize("v_mode", ["full", "t_only"])
def test_double_backward_decomposition(name, x_dim, cond_dim, out_dim, v_mode):
    params, x, cond, t, u, v = _problem(x_dim, cond_dim, out_dim)
    if v_mode == "t_only":
        v[:, :-1] = 0.0
    ref = torch_double_backward(params, x, cond, t, u, v)
    got = jet_double_backward(params, x, cond, t, u, v)
    assert len(ref) == len(got)
    labels = ["du"] + ["dx"] + (["dcond"] if cond is not None and cond.numel() else []) + ["dt"] + \
        [f"param{i}" for i in range(2 * len(params))]
    for lab, r, g in zip(labels, ref, got):
        r = torch.zeros_like(g) if r is None else r
        g = torch.zeros_like(r) if g is None else g
        scale = r.abs().max().clamp_min(1e-300)
        if lab == f"param{2 * len(params) - 1}":
            # the output-layer bias does not enter J: its gradient is exactly 0 in both statements
            assert r.abs().max().item() == 0.0 and g.abs().max().item() == 0.0, lab
            continue
        err = ((g - r).abs().max() / scale).item()
        assert err <= TOL, (name, v_mode, lab, err)
