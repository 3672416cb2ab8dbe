"""GPU tests of the MMD permutation test (csrc/dmip_mmd_test.cu) through dmip.metrics and the C ABI (pytest -m gpu).

Bar: every statistic within 1e-2 of the float64 null standard deviation of the same data (tests/mmd_perm_oracle.py on
the same label bits).  Kernel values are rounded to multiples of n_bw / 2047 before the (exact) tensor-core product, so
the error is measured against the spread the test has to resolve, not against the statistic's own size."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import mmd_perm_oracle as mpo

pytestmark = pytest.mark.gpu
DEV = "cuda"
REL = 1e-2


def _sets(n_obs, n, m, d, seed, shift=0.0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n_obs, n, d, generator=g)
    y = torch.randn(n_obs, m, d, generator=g) * 1.1 + shift
    return x, y


def _sigmas(nb, d):
    return [float(s) for s in np.geomspace(0.3, 3.0, nb) * d ** 0.5] if nb > 1 else [float(d ** 0.5)]


# (n, m, d, n_bw, P): (2, 3), (1000, 777), N = 161 and 259 (not multiples of 32 or 128), d = 1, 3, 5, 16, 1 and 8
# bandwidths, P = 1 and 254 (the maximum of one call)
CONFIGS = [(2, 3, 1, 1, 1), (2, 3, 3, 8, 254), (1000, 777, 3, 1, 254), (1000, 777, 5, 8, 1), (100, 61, 16, 8, 254),
           (130, 129, 1, 8, 254), (1000, 777, 16, 1, 254), (100, 61, 5, 1, 1)]


@pytest.mark.parametrize("n,m,d,nb,P", CONFIGS)
def test_statistics_and_p_values_match_the_float64_oracle(n, m, d, nb, P):
    from dmip import metrics
    x, y = _sets(1, n, m, d, seed=n + 7 * m + d)
    sig = _sigmas(nb, d)
    rng = np.random.default_rng(n * m + d)
    labels = mpo.random_labels(rng, 254, n, m)                 # the null spread comes from all 254
    ref = mpo.permutation_statistics(x[0].numpy(), y[0].numpy(), sig, labels)
    tol = REL * ref[1:].std()
    lab = torch.from_numpy(labels[None, :P].view(np.int32)).to(DEV)
    out, p = metrics.mmd2_permutation_statistics(x.to(DEV), y.to(DEV), sig, lab)
    got = out[0].cpu().numpy()
    err = np.abs(got - ref[:P + 1]).max()
    print(f"n={n} m={m} d={d} nb={nb} P={P}: max err / null std = {err / ref[1:].std():.2e}")
    assert err <= tol, (err, tol)
    direct = metrics.mmd2(x[0].to(DEV), y[0].to(DEV), sig).sum(-1).item()
    assert abs(got[0] - direct) <= tol, (got[0], direct, tol)
    p_ref = mpo.p_value(ref[0], ref[1:P + 1])
    slack = np.count_nonzero(np.abs(ref[1:P + 1] - ref[0]) <= tol) / (P + 1)
    assert abs(p[0].item() - p_ref) <= slack + 1e-15, (p[0].item(), p_ref, slack)
    assert p[0].item() == (1 + np.count_nonzero(got[1:] >= got[0])) / (P + 1)


def test_batching_determinism_launches_and_chunked_calls():
    from dmip import _lib, metrics
    x, y = _sets(4, 700, 450, 3, seed=3)
    x, y = x.to(DEV), y.to(DEV)
    sig = [0.8, 1.6]
    lab = metrics.permutation_labels(4, 700, 450, 200, generator=torch.Generator(device=DEV).manual_seed(1))
    a, pa = metrics.mmd2_permutation_statistics(x, y, sig, lab)
    assert _lib.lib().dmip_last_launch_count() == 2
    b, pb = metrics.mmd2_permutation_statistics(x, y, sig, lab)
    assert torch.equal(a, b) and torch.equal(pa, pb), "two runs differ"
    for o in range(4):
        s, ps = metrics.mmd2_permutation_statistics(x[o], y[o], sig, lab[o:o + 1])
        assert torch.equal(s[0], a[o]) and torch.equal(ps[0], pa[o]), o
    # the public entry: same generator state -> same labels -> same results; more than 254 permutations in two calls
    st, p, null = metrics.mmd2_test(x, y, sig, 200, generator=torch.Generator(device=DEV).manual_seed(1))
    assert torch.equal(st, a[:, 0]) and torch.equal(null, a[:, 1:]) and torch.equal(p, pa)
    st2, p2, null2 = metrics.mmd2_test(x, y, sig, 300, generator=torch.Generator(device=DEV).manual_seed(1))
    assert null2.shape == (4, 300) and (st2 - st).abs().max().item() <= 1e-9
    assert torch.equal(p2, (1 + (null2 >= st2[:, None]).sum(-1)).double() / 301)
    s1, p1, n1 = metrics.mmd2_test(x[0], y[0], sig, 17)
    assert s1.shape == () and p1.shape == () and n1.shape == (17,)


def test_bad_label_rows_give_nan():
    from dmip import metrics
    x, y = _sets(2, 40, 50, 2, seed=9)
    rng = np.random.default_rng(0)
    labels = np.stack([mpo.random_labels(rng, 6, 40, 50) for _ in range(2)])
    labels[1, 3, 0] ^= 4                                               # observation 1, permutation 3: 39 or 41 bits
    lab = torch.from_numpy(labels.view(np.int32)).to(DEV)
    out, p = metrics.mmd2_permutation_statistics(x.to(DEV), y.to(DEV), [1.0], lab)
    out = out.cpu().numpy()
    assert np.isnan(out[1, 4]) and np.isfinite(np.delete(out[1], 4)).all() and np.isfinite(out[0]).all()
    assert np.isfinite(p[0].item()) and np.isnan(p[1].item())
    ref = mpo.permutation_statistics(x[1].numpy(), y[1].numpy(), [1.0], labels[1])
    assert np.isnan(ref[4])


def test_guarded_buffers_and_c_level_errors():
    from dmip import metrics
    os.environ["DMIP_GUARD"] = "1"
    try:
        for (n, m, n_obs, d, nb, P) in [(2, 2, 1, 1, 1, 1), (3, 1027, 3, 3, 8, 254), (129, 130, 2, 16, 2, 17)]:
            x, y = _sets(n_obs, n, m, d, seed=n + m)
            metrics.mmd2_test(x.to(DEV), y.to(DEV), _sigmas(nb, d), P)   # Guarded.check raises on a canary hit
    finally:
        os.environ.pop("DMIP_GUARD", None)
    L = metrics._bind()
    x, y = torch.zeros(10, 3, device=DEV), torch.zeros(12, 3, device=DEV)
    lab = metrics.permutation_labels(1, 10, 12, 4)
    out = torch.full((64,), 7.0, dtype=torch.float64, device=DEV)
    keep = []

    def desc(**kw):
        d = metrics.DmipMmdTest()
        d.dim, d.n_obs, d.n, d.m, d.n_bw, d.n_perm = 3, 1, 10, 12, 1, 4
        d.sigma[0] = 1.0
        d.x, d.y, d.labels, d.out, d.p_value = x.data_ptr(), y.data_ptr(), lab.data_ptr(), out.data_ptr(), None
        for k, v in kw.items():
            if k == "sigma":
                d.sigma[0] = v
            else:
                setattr(d, k, v)
        nbytes = L.dmip_mmd_test_workspace_bytes(C.byref(d))
        ws = torch.empty(max(nbytes, 8), dtype=torch.uint8, device=DEV)
        keep.append(ws)
        d.workspace, d.workspace_bytes = ws.data_ptr(), nbytes
        return d

    for kw in (dict(dim=0), dict(dim=17), dict(n_obs=0), dict(n=1), dict(m=1), dict(n_bw=0), dict(n_bw=9),
               dict(sigma=0.0), dict(sigma=-2.0), dict(sigma=float("inf")), dict(sigma=float("nan")), dict(n_perm=0),
               dict(n_perm=255), dict(x=None), dict(y=None), dict(labels=None), dict(out=None),
               dict(labels=lab.data_ptr() + 2)):
        rc = L.dmip_mmd_test(C.byref(desc(**kw)), None)
        assert rc == -1 and L.dmip_last_error(), (kw, rc)
    big = desc(n=600000, m=600000)
    assert L.dmip_mmd_test_workspace_bytes(C.byref(big)) == 0
    big.workspace_bytes = 1 << 30
    assert L.dmip_mmd_test(C.byref(big), None) == -1 and b"pooled" in L.dmip_last_error()
    d = desc()
    d.workspace_bytes -= 8
    assert L.dmip_mmd_test(C.byref(d), None) == -3 and b"workspace" in L.dmip_last_error()
    torch.cuda.synchronize()
    assert (out == 7.0).all(), "a refused call wrote its output"
    assert L.dmip_mmd_test(C.byref(desc()), None) == 0                 # p_value NULL is allowed
    torch.cuda.synchronize()
    assert torch.isfinite(out[:5]).all() and (out[5:] == 7.0).all()


def test_calibration_under_h0_and_power():
    """200 tests of two N(0, I_3) draws of 512 (one batched call, fixed seeds): the rejection rate at alpha = 0.05 lies in
    the 99.9 % binomial interval of Binomial(200, 0.05).  A 0.25 sigma mean shift at n = m = 2048: p = 1/255."""
    from scipy.stats import binom
    from dmip import metrics
    g = torch.Generator(device=DEV).manual_seed(11)
    x = torch.randn(200, 512, 3, device=DEV, generator=g)
    y = torch.randn(200, 512, 3, device=DEV, generator=g)
    _, p, _ = metrics.mmd2_test(x, y, [3 ** 0.5], generator=g)
    rejections = int((p <= 0.05).sum().item())
    lo, hi = binom.interval(0.999, 200, 0.05)
    print(f"H0: {rejections} / 200 rejections at alpha = 0.05 (99.9 % interval {lo:.0f}..{hi:.0f})")
    assert lo <= rejections <= hi, (rejections, lo, hi)
    x = torch.randn(2048, 3, device=DEV, generator=g)
    y = torch.randn(2048, 3, device=DEV, generator=g) + torch.tensor([0.25, 0.0, 0.0], device=DEV)
    _, p, _ = metrics.mmd2_test(x, y, [3 ** 0.5], generator=g)
    assert p.item() == 1 / 255, p.item()


def test_bf16_and_fp32_posteriors_of_the_trained_linear_cde():
    """What the test is for: 2^16 bf16 against 2^16 fp32 samples of the trained linear CDE (200 steps, different Philox
    seeds) are not distinguishable at the 1 % level; the same sampler at two observations is, at p = 1/255."""
    import gpu_cases as gc
    from dmip import metrics
    model = gc.trained_model()
    N = 1 << 16
    draw = lambda yobs, prec, seed: model(torch.tensor(yobs), num_samples=N, num_steps=200, precision=prec, seed=seed,
                                          return_tensor=True)
    f32 = draw([0.4, -0.7], "fp32", 1)
    b16 = draw([0.4, -0.7], "bf16", 2)
    other = draw([-0.3, 0.5], "bf16", 3)
    bw = metrics.median_bandwidth(f32, b16)
    sig = [bw / 2, bw, 2 * bw]
    g = torch.Generator(device=DEV).manual_seed(5)
    st, p, null = metrics.mmd2_test(f32, b16, sig, generator=g)
    print(f"bf16 vs fp32, 2^16 each: MMD^2_u = {st.item():.3e}, null std {null.std().item():.3e}, p = {p.item():.4f}")
    st2, p2, _ = metrics.mmd2_test(b16, other, sig, generator=g)
    print(f"y = (0.4, -0.7) vs (-0.3, 0.5): MMD^2_u = {st2.item():.3e}, p = {p2.item():.4f}")
    assert p.item() >= 0.01
    assert p2.item() == 1 / 255
