"""The fused score-training losses across state dimension, net shape and batch tails, against the fp64 oracle
(pytest -m gpu).

The golden fixtures (tests/test_gpu_losses.py) check the loss kernels at d in {2, 3, 26}, two net shapes and batches
that fill every tile.  This sweep covers what the kernels claim beyond that:
  A  the state dimension d and the Score-FPE route: forward-only (second-order streams, d <= 4), the adjoint route
     (grad_x pass + reverse sweep: d = 5 ... 31, or forced with 'exact_adjoint') and Hutchinson; d = 32 must raise;
  B  net shapes on the FFMA kernels: 2 ... 8 Linear layers of widths 1 ... 512; width 513 and 9 layers must raise;
  C  the in/out width limit of the tcgen05 kernels (kTclSmallF = 64);
  D  every loss option at d = 2 and d = 4;
  E  PosteriorLoss at xdim = 1 ... 4 (xdim = 5 must raise).
Every case runs at batches that leave the last tile partial (B = 1, 37, 301; B <= 64 where the exact oracle carries
d(d+1)/2 second-order streams, d >= 26), under both kernel families, and checks which family ran."""
import pytest

import gpu_cases as gc

pytestmark = pytest.mark.gpu

H3 = (512, 512, 512)
BATCHES = (1, 37, 301)
BATCHES_WIDE = (1, 37)

# the compiled tcgen05 stream sets (has_I, has_T, n_tan, has_Q): mirrors DMIP_TCL_CONFIGS in csrc/dmip_tcl.cu
TCL_CONFIGS = {(0, 0, 0, 0), (0, 1, 0, 0), (1, 1, 0, 0), (0, 1, 2, 1), (1, 1, 2, 1), (1, 1, 3, 1), (1, 1, 4, 1),
               (0, 0, 3, 0)}
K_MAX_D = 4             # dmip_loss.cu kMaxD: largest d of the forward-only Score-FPE route
K_ROWS = 32             # dmip_tile.cuh kRows: stream rows per FFMA tile
K_TCL_WIN = 32          # dmip_tcl.h kTclWin: rows per tcgen05 epilogue window (two per 64-row tile)
K_TCL_SMALL_F = 64      # dmip_tcl.h kTclSmallF: largest in_dim / out_dim of the tcgen05 kernels

PINN_FPE = dict(lam=0.5, lam2=0.7, pde_loss="FPE", ic_metric="L2", pde_metric="L1")
DSMPDE_FPE = dict(lam=0.3, pde_loss="FPE", pde_metric="L2")
PINN_CFPE = dict(lam=0.01, lam2=0.7, pde_loss="cScoreFPE", ic_metric="L2", pde_metric="L2")
DSMPDE_CFPE = dict(lam=0.05, pde_loss="cScoreFPE", pde_metric="L1")


def _loss(group, model, xdim, ydim, kind, kw=None, hidden=H3, batches=None):
    d = xdim if model == "CDE" else xdim + ydim
    return dict(group=group, model=model, xdim=xdim, ydim=ydim, hidden=tuple(hidden), kind=kind, kw=dict(kw or {}),
                batches=batches or (BATCHES_WIDE if d >= 26 else BATCHES))


def _hid(h):
    return "x".join(map(str, h)) if len(set(h)) > 1 else f"{h[0]}^{len(h)}"


LOSS_SWEEP = {}
# A. state dimension x Score-FPE route, [512]^3
for d in (1, 2, 3, 4):
    for route in ("exact", "exact_adjoint"):
        LOSS_SWEEP[f"A-cde{d}-pinn-{route}"] = _loss("A", "CDE", d, 3, "PINN", dict(PINN_FPE, divergence_method=route))
        LOSS_SWEEP[f"A-cde{d}-dsmpde-{route}"] = _loss("A", "CDE", d, 3, "DSM_PDE",
                                                      dict(DSMPDE_FPE, divergence_method=route))
for d in (1, 4):
    LOSS_SWEEP[f"A-cde{d}-pinn-hutchinson"] = _loss("A", "CDE", d, 3, "PINN", dict(PINN_FPE, divergence_method="hutchinson"))
    LOSS_SWEEP[f"A-cde{d}-dsmpde-hutchinson"] = _loss("A", "CDE", d, 3, "DSM_PDE",
                                                     dict(DSMPDE_FPE, divergence_method="hutchinson"))
LOSS_SWEEP["A-cde5-pinn-exact"] = _loss("A", "CDE", 5, 3, "PINN", PINN_FPE)
LOSS_SWEEP["A-cde5-dsmpde-exact"] = _loss("A", "CDE", 5, 3, "DSM_PDE", DSMPDE_FPE)
LOSS_SWEEP["A-cdiffe2+29-pinn-exact"] = _loss("A", "CDiffE", 2, 29, "PINN", PINN_FPE)
LOSS_SWEEP["A-cdiffe2+29-dsmpde-exact"] = _loss("A", "CDiffE", 2, 29, "DSM_PDE", DSMPDE_FPE)
# B. net shapes (FFMA kernels), CDE d = 2
for h in ((1,), (7, 129), (128, 128, 127), (33, 1, 100, 7), (512, 64, 512), (16,) * 7):
    LOSS_SWEEP[f"B-{_hid(h)}-pinn-exact"] = _loss("B", "CDE", 2, 3, "PINN", PINN_FPE, hidden=h)
    LOSS_SWEEP[f"B-{_hid(h)}-dsm"] = _loss("B", "CDE", 2, 3, "DSM", hidden=h)
# C. the tcgen05 in/out width limit: in_dim 64 (tcgen05) / 65 (FFMA); out_dim 63
for ydim in (61, 62):
    LOSS_SWEEP[f"C-cde2+{ydim}-dsm"] = _loss("C", "CDE", 2, ydim, "DSM")
    LOSS_SWEEP[f"C-cde2+{ydim}-pinn-cscorefpe"] = _loss("C", "CDE", 2, ydim, "PINN", PINN_CFPE)
LOSS_SWEEP["C-cdiffe2+61-pinn-hutchinson"] = _loss("C", "CDiffE", 2, 61, "PINN", dict(PINN_FPE, divergence_method="hutchinson"))
LOSS_SWEEP["C-cdiffe2+61-dsmpde-hutchinson"] = _loss("C", "CDiffE", 2, 61, "DSM_PDE",
                                                    dict(DSMPDE_FPE, divergence_method="hutchinson"))
# D. every loss option at d = 2 and d = 4 (the PINN ic L2 / pde L1 and DSM_PDE FPE L2 cases are in A)
for d in (2, 4):
    LOSS_SWEEP[f"D-cde{d}-dsm"] = _loss("D", "CDE", d, 3, "DSM")
    LOSS_SWEEP[f"D-cde{d}-dsmpde-fpe-l1"] = _loss("D", "CDE", d, 3, "DSM_PDE", dict(DSMPDE_FPE, pde_metric="L1"))
    LOSS_SWEEP[f"D-cde{d}-dsmpde-cscorefpe-l1"] = _loss("D", "CDE", d, 3, "DSM_PDE", DSMPDE_CFPE)
    for ic, pde in (("L1", "L1"), ("L1", "L2"), ("L2", "L2")):
        LOSS_SWEEP[f"D-cde{d}-pinn-ic{ic}-pde{pde}"] = _loss("D", "CDE", d, 3, "PINN",
                                                            dict(PINN_FPE, ic_metric=ic, pde_metric=pde))
    LOSS_SWEEP[f"D-cde{d}-pinn-cscorefpe"] = _loss("D", "CDE", d, 3, "PINN", PINN_CFPE)
    LOSS_SWEEP[f"D-cde{d}-pinn2-fpe"] = _loss("D", "CDE", d, 3, "PINN2", dict(lam=0.5, lam2=0.7, pde_loss="FPE",
                                                                           ic_metric="L2"))
    LOSS_SWEEP[f"D-cde{d}-pinn2-cscorefpe"] = _loss("D", "CDE", d, 3, "PINN2", dict(lam=0.01, lam2=0.7,
                                                                                 pde_loss="cScoreFPE", ic_metric="L1"))

POSTERIOR_SWEEP = {f"E-xdim{x}-{_hid(h)}": dict(group="E", xdim=x, ydim=23, hidden=h, batches=BATCHES)
                   for x in (1, 2, 3, 4) for h in (H3, (64, 64))}

# shapes outside the documented limits: (case, substring of the error)
REJECTED = {
    "A-cdiffe2+30-pinn-exact": (_loss("A", "CDiffE", 2, 30, "PINN", PINN_FPE), "too many jet streams"),
    "A-cdiffe2+30-dsmpde-exact": (_loss("A", "CDiffE", 2, 30, "DSM_PDE", DSMPDE_FPE), "too many jet streams"),
    "B-513-pinn-exact": (_loss("B", "CDE", 2, 3, "PINN", PINN_FPE, hidden=(513,)), "bad width"),
    "B-513-dsm": (_loss("B", "CDE", 2, 3, "DSM", hidden=(64, 513)), "bad width"),
    "B-9layers-pinn-exact": (_loss("B", "CDE", 2, 3, "PINN", PINN_FPE, hidden=(16,) * 8), "at most 8 Linear layers"),
    "B-9layers-dsm": (_loss("B", "CDE", 2, 3, "DSM", hidden=(16,) * 8), "at most 8 Linear layers"),
}
POSTERIOR_REJECTED = {"E-xdim5": (dict(group="E", xdim=5, ydim=23, hidden=H3), "1 <= xdim <= 4")}


# ------------------------------------------------------------------------------------------- dispatch table
def passes(c):
    """the kernel passes one fused call runs: (has_I, has_T, n_tan, has_Q, grad_x pass?, in_dim, out_dim, hidden)
    — the stream sets cfg_from_loss / plan_loss / plan_posterior in csrc/dmip_loss.cu build"""
    if "kind" not in c:                                             # PosteriorLoss: prior net (Jacobian), likelihood net
        x, y = c["xdim"], c["ydim"]
        return [(0, 0, x, 0, False, x + 1, x, c["hidden"]), (0, 0, 0, 0, False, x + y + 1, x, c["hidden"])]
    d = c["xdim"] if c["model"] == "CDE" else c["xdim"] + c["ydim"]
    io = (c["xdim"] + c["ydim"] + 1, d, c["hidden"])
    kind, kw = c["kind"], c["kw"]
    if kind == "DSM":
        return [(0, 0, 0, 0, False) + io]
    has_i = int(kind in ("PINN", "PINN2"))
    if kw.get("pde_loss", "FPE") != "FPE":
        return [(has_i, 1, 0, 0, False) + io]
    div = kw.get("divergence_method", "exact")
    if div == "exact" and d <= K_MAX_D:                             # forward-only: tangents S_k and pairs Q_ik
        return [(has_i, 1, d, 1, False) + io]
    n_tan = 1 if div in ("hutchinson", "approx", "approximate") else d
    return [(0, 0, n_tan, 0, True) + io, (has_i, 1, 0, 0, False) + io]   # grad_x pass, then the main pass


def on_tcgen05(p):
    """plan_tcl: [in <= 64] -> 512 -> 512 -> 512 -> [out <= 64], a compiled stream set, not the grad_x pass"""
    i, t, n, q, gx, in_dim, out_dim, hidden = p
    return (not gx and hidden == H3 and in_dim <= K_TCL_SMALL_F and out_dim <= K_TCL_SMALL_F
            and (i, t, n, q) in TCL_CONFIGS)


def n_streams(p):
    i, t, n, q = p[:4]
    return 1 + i + t + n + (n * (n + 1) // 2 if q else 0)


def spt(p, family):
    """samples per tile (forward, backward) of a pass: FFMA kRows / streams; tcgen05 2 (kTclWin / streams)"""
    n_adj = 1 + p[0] + p[1]
    if p[4]:                                                        # grad_x pass: its reverse sweep carries P | S_k too
        n_adj = n_streams(p)
    if family == "ffma":
        return K_ROWS // n_streams(p), K_ROWS // n_adj
    return 2 * (K_TCL_WIN // n_streams(p)), 2 * (K_TCL_WIN // n_adj)


ALL = {**LOSS_SWEEP, **POSTERIOR_SWEEP}


# ------------------------------------------------------------------------------------------- tests
def _ok(res):
    err, tol, extra = res
    assert err <= tol, (err, tol, extra)


@pytest.fixture(params=["tc", "ffma"])
def loss_path(request, monkeypatch):
    """'tc' = the tcgen05 kernels wherever plan_tcl selects them (the default), 'ffma' = the fp32 FFMA kernels forced for
    every pass"""
    monkeypatch.setenv("DMIP_LOSS_PATH", request.param)
    return request.param


@pytest.mark.parametrize("loss_path", ["tc", "ffma"], indirect=True)     # innermost: the two runs of a case in a row
@pytest.mark.parametrize("name", sorted(LOSS_SWEEP))                     # share its oracle results
def test_fused_loss_sweep(name, loss_path):
    c = LOSS_SWEEP[name]
    _ok(gc.case_loss_sweep(c["model"], c["xdim"], c["ydim"], c["hidden"], c["kind"], c["kw"], c["batches"]))


@pytest.mark.parametrize("loss_path", ["tc", "ffma"], indirect=True)
@pytest.mark.parametrize("name", sorted(POSTERIOR_SWEEP))
def test_posterior_loss_sweep(name, loss_path):
    c = POSTERIOR_SWEEP[name]
    _ok(gc.case_posterior_loss_sweep(c["xdim"], c["hidden"], c["batches"], ydim=c["ydim"]))


@pytest.mark.parametrize("name", sorted(REJECTED))
def test_shapes_beyond_the_limits_raise(name, loss_path):
    c, match = REJECTED[name]
    _ok(gc.case_loss_rejected(c["model"], c["xdim"], c["ydim"], c["hidden"], c["kind"], c["kw"], match))


@pytest.mark.parametrize("name", sorted(POSTERIOR_REJECTED))
def test_posterior_loss_beyond_the_limits_raises(name, loss_path):
    c, match = POSTERIOR_REJECTED[name]
    _ok(gc.case_posterior_loss_rejected(c["xdim"], c["hidden"], match, ydim=c["ydim"]))


@pytest.mark.parametrize("name", sorted(ALL))
def test_the_kernel_family_that_runs_is_the_one_the_table_names(name):
    """a pass on the tcgen05 kernels launches pack + forward + backward + 4 weight-gradient GEMMs = 7 kernels, the same
    pass on the FFMA kernels 4 transposes + forward + backward + 4 weight-gradient kernels = 10; every other launch
    (grad_x pass, surrogate, target assembly) is the same under both.  So forcing DMIP_LOSS_PATH=ffma adds exactly 3
    launches per pass the table puts on tcgen05, and none where it names none: a case meant for the tensor-core kernels
    cannot silently test the FFMA kernels twice."""
    c = ALL[name]
    if "kind" in c:
        counts = gc.case_loss_launches(c["model"], c["xdim"], c["ydim"], c["hidden"], c["kind"], c["kw"])
    else:
        counts = gc.case_posterior_loss_launches(c["xdim"], c["hidden"], ydim=c["ydim"])
    n_tc = sum(on_tcgen05(p) for p in passes(c))
    assert counts["ffma"] - counts["tc"] == 3 * n_tc, (counts, n_tc)


def test_every_compiled_tcgen05_stream_set_is_swept():
    reached = {p[:4] for c in ALL.values() for p in passes(c) if on_tcgen05(p)}
    assert reached == TCL_CONFIGS, TCL_CONFIGS - reached


def test_the_sweep_reaches_the_documented_limits():
    dims = {c["xdim"] if c["model"] == "CDE" else c["xdim"] + c["ydim"] for c in LOSS_SWEEP.values()}
    assert {1, 2, 3, 4, 5, 31} <= dims
    assert {c["xdim"] + c["ydim"] for c, _ in REJECTED.values() if c["model"] == "CDiffE"} == {32}
    assert {c["xdim"] for c in POSTERIOR_SWEEP.values()} == {1, 2, 3, 4}
    assert {len(c["hidden"]) + 1 for c in LOSS_SWEEP.values()} >= {2, 3, 4, 5, 8}


@pytest.mark.parametrize("group", "ABCDE")
def test_every_group_leaves_a_partial_last_tile_in_both_families(group):
    """in each group some batch leaves the last forward tile and the last backward tile partial, on the FFMA kernels and
    (where the group has tcgen05 passes) on the tcgen05 kernels — a dropped, doubled or misread tail sample shows"""
    cases = [c for c in ALL.values() if c["group"] == group]
    for family in ("ffma", "tc"):
        runs = [(p, B) for c in cases for p in passes(c) for B in c["batches"] if family == "ffma" or on_tcgen05(p)]
        if family == "tc" and group == "B":
            assert not runs                                         # group B is the FFMA net-shape sweep
            continue
        assert any(B % spt(p, family)[0] for p, B in runs), (group, family, "forward")
        assert any(B % spt(p, family)[1] for p, B in runs), (group, family, "backward")
