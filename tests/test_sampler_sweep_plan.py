"""The case table of the sampler / forward sweep (tests/test_gpu_sampler_sweep.py) and what it must cover, checked
without a GPU.

The fused sampler k_tc_mlp (csrc/dmip_tc.cu) is compiled as 10 instantiations <NP, VAR, L0TMEM>: NP = state pieces of
8 columns a row may hold (1, 4 or 13), VAR = CDE / CDiffE / DPS, L0TMEM = the layer-0 operand is one f16 part in tensor
memory instead of shared memory.  The forward (dmip_mlp_forward) runs <1, CDE, false> in forward mode.  Shapes the
tensor-core kernels do not serve go to the FFMA kernels (csrc/dmip_f32.cu), and the Python classes make that switch
silently (only `last_precision` records it).  This file
  * restates the dispatch (launch() / launch_sampler_tc() / tc_net_geom() and the Python fallback) as a table, and
    checks it against the instantiations dmip_tc.cu compiles;
  * asserts that the sweep reaches every instantiation, every split of the state pieces over the four column groups,
    and every tile tail (lone particle, partial tile, masked CTA of the last pair, a pair across two observations);
  * runs the fp64 oracle with plausible kernel bugs injected and asserts each misses the bf16 bound by >= 5x, so the
    sweep can fail;
  * pins the tcgen05 packing limits at the C ABI (dmip_pack_bytes needs no device)."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

import gpu_cases as gc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
H3 = (512, 512, 512)
K_TILE_M = 128          # dmip_tc.cu kTileM: particles per tcgen05 tile
K_CLUSTER = 2           # dmip_tc.cu kCluster: CTAs per cluster, one tile each per round
K_ROWS = 32             # dmip_tile.cuh kRows: particles per FFMA tile
N_SM_NOMINAL = 148      # B200 SM count, for the CPU-side plan only: the GPU cases read it from the device
FFMA = "FFMA"

# ------------------------------------------------------------------------------------------- dispatch mirror
# launch() in csrc/dmip_tc.cu: (variant, largest xdim of the row, NP), tested in this order.  The last row of each
# variant is also the xdim limit of launch_sampler_tc() (and of the Python fallback condition, models/diffusion.py).
NP_TABLE = [("CDE", 8, 1), ("CDE", 32, 4), ("CDE", 104, 13),
            ("CDiffE", 8, 1), ("CDiffE", 32, 4),
            ("DPS", 8, 1)]
TC_YDIM_MAX = {"CDiffE": 24}                  # launch_sampler_tc: the CDiffE y quads cgp and cgp + 4
FORWARD_INST = ("forward", 1, "CDE", False)   # launch_forward_tc -> launch(): state_cols = 1, never l0_tmem


def _up(v, m):
    return (v + m - 1) // m * m


def k0pad(n_varying, split):
    """tc_net_geom: layer-0 GEMM depth; l0_split 4 is one f16 part, 2 / 3 add a lo part of x (and of W0)"""
    parts = 1 if split == 4 else split
    return _up((parts - 1) * _up(n_varying, 8) + n_varying, 16)


def net_on_tc(hidden, out_dim, n_varying, split):
    """_lib.tc_supported / tc_net_geom: [in] -> 512 -> 512 -> 512 -> [out <= 128], layer-0 depth <= 512"""
    return tuple(hidden) == H3 and out_dim <= 128 and k0pad(n_varying, split) <= 512


def l0_tmem(variant, n_varying, split):
    """launch_sampler_tc: one f16 part of <= 128 k, whole 8-element state pieces (not CDiffE: y_t sits beside x)"""
    return split == 4 and variant != "CDiffE" and k0pad(n_varying, split) <= 128


def sampler_inst(variant, xdim, ydim, hidden, l0_split):
    """(NP, VAR, L0TMEM) of k_tc_mlp that precision='bf16' runs, or FFMA where the Python classes fall back"""
    dv = xdim + ydim if variant == "CDiffE" else xdim
    out_dim = xdim + ydim if variant == "CDiffE" else xdim
    if not net_on_tc(hidden, out_dim, dv, l0_split):
        return FFMA
    if variant == "DPS" and not net_on_tc(hidden, xdim, xdim, l0_split):      # the prior net
        return FFMA
    if ydim > TC_YDIM_MAX.get(variant, ydim):
        return FFMA
    for v, xmax, np_ in NP_TABLE:
        if v == variant and xdim <= xmax:
            return (np_, variant, l0_tmem(variant, dv, l0_split))
    return FFMA


def forward_inst(in_dim, out_dim, hidden, l0_split):
    return FORWARD_INST if net_on_tc(hidden, out_dim, in_dim, l0_split) else FFMA


def compiled_instantiations():
    """the k_tc_mlp<NP, VAR, L0TMEM> instantiations init_device() prepares (one per launch() branch)"""
    src = open(os.path.join(ROOT, "diffusion-modelling-for-inverse-problems_b200", "csrc", "dmip_tc.cu")).read()
    names = {"CDE": "CDE", "CDIFFE": "CDiffE", "DPS": "DPS"}
    return {(int(n), names[v], b == "true")
            for n, v, b in re.findall(r"DMIP_SET_SMEM\((\d+), DMIP_(CDE|CDIFFE|DPS), (true|false)\);", src)}


# ------------------------------------------------------------------------------------------- the sweep
TAILS = ((1, 1), (3, 300))      # a lone particle; 3 observations x 300: partial tiles, 9 tiles, pairs across observations
FFMA_RUNS = ((1, 1), (1, 31), (1, 33), (3, 300))


def _s(group, variant, xdim, ydim, inst, hidden=H3, l0_split=4, S=5, runs=TAILS, seed=0, y_scale=10.0, **kw):
    """y_scale: observations ~ N(0, 10^2), far enough from the origin that one y column left out of the layer-0 bias
    moves the samples past the bound (test_injected_sampler_bugs_miss_the_bf16_bound)"""
    return dict(group=group, variant=variant, xdim=xdim, ydim=ydim, hidden=tuple(hidden), l0_split=l0_split, S=S,
                runs=runs, seed=seed, inst=inst, y_scale=y_scale, **kw)


def _hid(h):
    return "x".join(map(str, h)) if len(set(h)) > 1 else f"{h[0]}^{len(h)}"


SAMPLER_SWEEP = {}
# A. CDE on tcgen05: state width x instantiation, l0_split 4; ydim across 1 ... 300.  xdim: (ydim, NP it runs)
A_CASES = {1: (1, 1), 7: (3, 1), 8: (27, 1), 9: (300, 4), 16: (1, 4), 17: (3, 4), 31: (27, 4), 32: (300, 4),
           33: (1, 13), 41: (3, 13), 56: (27, 13), 64: (300, 13), 97: (1, 13), 103: (3, 13), 104: (300, 13)}
for x, (yd, np_) in A_CASES.items():
    SAMPLER_SWEEP[f"A-cde{x}+{yd}"] = _s("A", "CDE", x, yd, (np_, "CDE", True), seed=x, guard=(x == 104))
# the shared-memory layer-0 operand at every NP
for x, splits, np_ in ((8, (2,), 1), (32, (2,), 4), (104, (2,), 13), (17, (1, 3), 4), (64, (1, 3), 13)):
    for sp in splits:
        SAMPLER_SWEEP[f"A-cde{x}+3-split{sp}"] = _s("A", "CDE", x, 3, (np_, "CDE", False), l0_split=sp, seed=50 + x)
# C. CDiffE on tcgen05: the y quads cgp / cgp + 4, ydim not a multiple of 4
for x, yd in ((1, 1), (2, 24), (8, 7), (9, 24), (16, 13), (32, 1), (32, 24)):
    for sp in (4, 2):
        SAMPLER_SWEEP[f"C-cdiffe{x}+{yd}-split{sp}"] = _s("C", "CDiffE", x, yd, (1 if x <= 8 else 4, "CDiffE", False),
                                                         l0_split=sp, seed=100 + x + yd, guard=(x, yd, sp) == (9, 24, 4))
# y reaches a CDiffE net only through y_t = alpha(tau) y + std(tau) eta, and the default init (gain 1) shrinks every
# hidden layer's signal by about 1/sqrt(3): with gain 2 a wrong y column or re-diffusion draw shows in the samples
SAMPLER_SWEEP["C-cdiffe9+24-split4-gain2"] = _s("C", "CDiffE", 9, 24, (4, "CDiffE", False), seed=133, gain=2.0)
# D. DPS on tcgen05: two nets per pass
for x in (1, 5, 8):
    for yd in (1, 23, 200):
        for sp in (4, 2):
            SAMPLER_SWEEP[f"D-dps{x}+{yd}-split{sp}"] = _s("D", "DPS", x, yd, (1, "DPS", sp == 4), l0_split=sp,
                                                          seed=200 + x + yd, guard=(x, yd, sp) == (8, 200, 4))
# E. the FFMA sampler (precision 'fp32'; 'bf16' must fall back to it): net shapes, and states past the tcgen05 limits
for h in ((64, 64), (7, 129), (33, 1, 100, 7), (16,) * 7):
    for v in ("CDE", "CDiffE", "DPS"):
        SAMPLER_SWEEP[f"E-{v.lower()}3+5-{_hid(h)}"] = _s("E", v, 3, 5, FFMA, hidden=h, runs=FFMA_RUNS, seed=300,
                                                         fp32=True, guard=(v, h) == ("DPS", (33, 1, 100, 7)))
for x in (105, 128, 300):
    SAMPLER_SWEEP[f"E-cde{x}+3"] = _s("E", "CDE", x, 3, FFMA, runs=FFMA_RUNS, seed=300 + x, fp32=True)
for x, yd in ((33, 25), (40, 100)):
    SAMPLER_SWEEP[f"E-cdiffe{x}+{yd}"] = _s("E", "CDiffE", x, yd, FFMA, runs=FFMA_RUNS, seed=300 + x, fp32=True)
for x in (9, 128):
    SAMPLER_SWEEP[f"E-dps{x}+3"] = _s("E", "DPS", x, 3, FFMA, runs=FFMA_RUNS, seed=400 + x, fp32=True)
# G. the in-kernel Philox stream against its injected mirror, and the VE-SDE with a corrector, at the new widths
for x, np_ in ((17, 4), (64, 13)):
    SAMPLER_SWEEP[f"G-cde{x}+3-philox"] = _s("G", "CDE", x, 3, (np_, "CDE", True), seed=500 + x, philox=True, fp32=True,
                                            guard=(x == 64))
    SAMPLER_SWEEP[f"G-cde{x}+3-ve-corrector"] = _s("G", "CDE", x, 3, (np_, "CDE", True), seed=600 + x, sde="VE", n_corr=1,
                                                  fp32=True)
SAMPLER_SWEEP["G-cdiffe9+24-philox"] = _s("G", "CDiffE", 9, 24, (4, "CDiffE", False), seed=509, philox=True, fp32=True)

# B. persistent tiles: (2 n_sm + 3) * 128 - 50 particles, tcgen05 against FFMA on the same noise (runs: see gpu_cases)
PERSISTENT = {
    "B-cde33+3": _s("B", "CDE", 33, 3, (13, "CDE", True), S=3, runs=None, seed=700, guard=True),
    "B-cde104+3": _s("B", "CDE", 104, 3, (13, "CDE", True), S=3, runs=None, seed=701),
    "B-cdiffe17+5": _s("B", "CDiffE", 17, 5, (4, "CDiffE", False), S=3, runs=None, seed=702),
    "B-dps8+23": _s("B", "DPS", 8, 23, (1, "DPS", True), S=3, runs=None, seed=703),
}


def _f(in_dim, out_dim, inst, hidden=H3, l0_split=4, cls="MLP", ns=(1, 127, 129, 300), scale=1.0, seed=0):
    return dict(group="F", in_dim=in_dim, out_dim=out_dim, hidden=tuple(hidden), l0_split=l0_split, cls=cls,
                ns=tuple(ns), scale=scale, seed=seed, inst=inst)


FORWARD_SWEEP = {}
# F. the tcgen05 forward: a covering set of in_dim x out_dim, inputs at scale 1 and 30
# (a bf16 forward is accurate to about 1e-3 absolute.  An MLP on two inputs runs its tanh layers unsaturated, so their
# bf16 rounding alone exceeds the bound — test_forward_cases_meet_the_bound_under_the_kernels_rounding — and in_dim 2
# is the MLP2 net below, whose one output also covers out_dim 1 with in_dim 512)
for i, (ind, outd) in enumerate(((64, 15), (65, 17), (128, 64), (129, 127), (256, 128), (512, 1), (512, 128))):
    for scale in (1.0, 30.0):
        FORWARD_SWEEP[f"F-{ind}to{outd}-x{scale:g}"] = _f(ind, outd, FORWARD_INST, scale=scale, seed=800 + i)
FORWARD_SWEEP["F-129to64-multiround"] = _f(129, 64, FORWARD_INST, ns=(300, "multi"), scale=30.0, seed=820)
FORWARD_SWEEP["F-mlp2-65to64"] = _f(65, 64, FORWARD_INST, cls="MLP2", scale=30.0, seed=821)
FORWARD_SWEEP["F-mlp2-2to1"] = _f(2, 1, FORWARD_INST, cls="MLP2", seed=822)
# each l0_split at its layer-0 depth limit, and one past it (falls back).  Inputs at scale 1: l0_split 1 rounds x and
# 2 rounds W0 to bf16, so their layer-0 error grows with |x| by design (4, the default, is the scale-30 sweep above)
for sp, lim in ((1, 512), (2, 256), (3, 168)):
    FORWARD_SWEEP[f"F-{lim}to17-split{sp}"] = _f(lim, 17, FORWARD_INST, l0_split=sp, seed=830 + sp)
    if sp != 1:                                   # in_dim 513 is past the FFMA kernels' width limit too
        FORWARD_SWEEP[f"F-{lim + 1}to17-split{sp}"] = _f(lim + 1, 17, FFMA, l0_split=sp, seed=840 + sp)
# the FFMA forward: 8 layers, a width-1 layer, in_dim 512, out_dim past 128
FORWARD_SWEEP["F-ffma-8layers"] = _f(9, 5, FFMA, hidden=(64,) * 7, seed=850)
FORWARD_SWEEP["F-ffma-width1"] = _f(9, 5, FFMA, hidden=(64, 1, 64), seed=851)
FORWARD_SWEEP["F-ffma-512to7"] = _f(512, 7, FFMA, hidden=(256, 128), scale=30.0, seed=852)
for outd in (129, 300):
    FORWARD_SWEEP[f"F-ffma-65to{outd}"] = _f(65, outd, FFMA, seed=853 + outd)

# H. descriptors the C ABI refuses (DMIP_EINVAL): (DmipSampler fields, substring of the message)
ABI_REJECTED = {
    "H-tc-cde105": (dict(variant="CDE", precision="bf16", xdim=105, ydim=3, hidden=H3), "xdim <= 104"),
    "H-tc-cdiffe33": (dict(variant="CDiffE", precision="bf16", xdim=33, ydim=3, hidden=H3), "xdim <= 32, ydim <= 24"),
    "H-tc-cdiffe-ydim25": (dict(variant="CDiffE", precision="bf16", xdim=3, ydim=25, hidden=H3), "xdim <= 32, ydim <= 24"),
    "H-tc-dps9": (dict(variant="DPS", precision="bf16", xdim=9, ydim=3, hidden=H3), "xdim <= 8"),
    "H-ffma-dps129": (dict(variant="DPS", precision="fp32", xdim=129, ydim=3, hidden=(16, 16)), "xdim <= 128"),
    "H-ffma-9layers": (dict(variant="CDE", precision="fp32", xdim=3, ydim=3, hidden=(16,) * 8), "n_layers 9 out of range"),
    "H-ffma-width513": (dict(variant="CDE", precision="fp32", xdim=3, ydim=3, hidden=(513,)), "width 513 out of range"),
}


def sampler_paths(c):
    """precision requested -> the path that must run ('bf16' = tcgen05, 'fp32' = FFMA)"""
    p = {"bf16": "fp32" if c["inst"] == FFMA else "bf16"}
    if c.get("fp32"):
        p["fp32"] = "fp32"
    return p


def forward_paths(c):
    return {"bf16": "fp32" if c["inst"] == FFMA else "bf16", "fp32": "fp32"}


def persistent_n(n_sm=N_SM_NOMINAL):
    return (2 * n_sm + 3) * K_TILE_M - 50


def _runs(c):
    return ((1, persistent_n()),) if c["runs"] is None else c["runs"]


ALL_SAMPLER = {**SAMPLER_SWEEP, **PERSISTENT}


# ------------------------------------------------------------------------------------------- tests: the table
def test_the_mirror_names_exactly_the_compiled_instantiations():
    mirror = {(np_, v, t) for v, _, np_ in NP_TABLE for t in (False, True)
              if not (t and v == "CDiffE")}
    assert mirror == compiled_instantiations()
    assert len(mirror) == 10


@pytest.mark.parametrize("name", sorted(ALL_SAMPLER))
def test_each_sampler_case_runs_the_instantiation_it_states(name):
    c = ALL_SAMPLER[name]
    assert sampler_inst(c["variant"], c["xdim"], c["ydim"], c["hidden"], c["l0_split"]) == c["inst"]


@pytest.mark.parametrize("name", sorted(FORWARD_SWEEP))
def test_each_forward_case_runs_the_instantiation_it_states(name):
    c = FORWARD_SWEEP[name]
    assert forward_inst(c["in_dim"], c["out_dim"], c["hidden"], c["l0_split"]) == c["inst"]


def test_every_instantiation_is_reached():
    reached = {c["inst"] for c in ALL_SAMPLER.values()} - {FFMA}
    assert reached == compiled_instantiations(), compiled_instantiations() - reached
    assert FORWARD_INST in {c["inst"] for c in FORWARD_SWEEP.values()}
    assert FFMA in {c["inst"] for c in FORWARD_SWEEP.values()}


def test_every_split_of_the_state_pieces_is_reached():
    """n_own / piece_lo split ceil(xdim / 8) pieces over four column groups: every residue mod 4 an NP admits, with a
    partial last piece and a whole one"""
    for np_, want in ((4, {0, 2, 3}), (13, {0, 1, 2, 3})):
        xs = {c["xdim"] for c in ALL_SAMPLER.values() if c["inst"] != FFMA and c["inst"][0] == np_}
        assert {(-(-x // 8)) % 4 for x in xs} == want, (np_, sorted(xs))
        assert any(x % 8 for x in xs) and any(x % 8 == 0 for x in xs), (np_, sorted(xs))


def _tails(n_obs, n_per_obs, tile, pair):
    tiles_per_obs = -(-n_per_obs // tile)
    n_tiles = n_obs * tiles_per_obs
    out = set()
    if n_obs * n_per_obs == 1:
        out.add("lone particle")
    if n_per_obs % tile:
        out.add("partial last tile")
    if pair:
        if n_tiles % K_CLUSTER:
            out.add("masked CTA in the last pair")
        if any((t // tiles_per_obs) != ((t + 1) // tiles_per_obs) for t in range(0, n_tiles - 1, K_CLUSTER)):
            out.add("pair across observations")
    return out


TC_TAILS = {"lone particle", "partial last tile", "masked CTA in the last pair", "pair across observations"}


@pytest.mark.parametrize("inst", sorted(compiled_instantiations(), key=str))
def test_every_instantiation_meets_every_tile_tail(inst):
    got = set()
    for c in ALL_SAMPLER.values():
        if c["inst"] == inst:
            for n_obs, n in _runs(c):
                got |= _tails(n_obs, n, K_TILE_M, True)
    assert got == TC_TAILS, TC_TAILS - got


def test_the_forward_meets_every_tile_tail():
    got = set()
    for c in FORWARD_SWEEP.values():
        if c["inst"] == FORWARD_INST:
            for n in c["ns"]:
                got |= _tails(1, persistent_n() if n == "multi" else n, K_TILE_M, True)
    assert {"lone particle", "partial last tile", "masked CTA in the last pair"} <= got


def test_persistent_cases_give_every_cta_two_tiles_and_a_partial_last_round():
    for n_sm in (N_SM_NOMINAL, 132, 160):                  # whatever the device, the formula keeps its promise
        n_tiles = -(-persistent_n(n_sm) // K_TILE_M)
        assert n_tiles >= 2 * n_sm and n_tiles % n_sm and n_tiles % K_CLUSTER
        assert persistent_n(n_sm) % K_TILE_M
    assert {c["variant"] for c in PERSISTENT.values()} == {"CDE", "CDiffE", "DPS"}


def test_the_ffma_cases_leave_a_partial_32_row_tile():
    for group in ("E",):
        runs = [r for c in SAMPLER_SWEEP.values() if c["group"] == group for r in c["runs"]]
        assert any(n % K_ROWS for _, n in runs) and any(n > K_ROWS for _, n in runs)
    for c in SAMPLER_SWEEP.values():
        if c["inst"] == FFMA:
            assert "fp32" in sampler_paths(c) and sampler_paths(c)["bf16"] == "fp32"


def test_the_sweep_reaches_the_documented_limits():
    tc = [c for c in ALL_SAMPLER.values() if c["inst"] != FFMA]
    ffma = [c for c in ALL_SAMPLER.values() if c["inst"] == FFMA]
    for v, xmax, _ in NP_TABLE:                     # each row's largest xdim is run on tcgen05, one past it is not
        assert any(c["variant"] == v and c["xdim"] == xmax for c in tc), (v, xmax)
        nxt = [r for r in NP_TABLE if r[0] == v and r[1] > xmax]
        if not nxt:
            assert sampler_inst(v, xmax + 1, 3, H3, 4) == FFMA
            assert any(c["variant"] == v and c["xdim"] > xmax and c["hidden"] == H3 for c in ffma), v
    assert any(c["variant"] == "CDiffE" and c["ydim"] == 24 for c in tc)
    assert any(c["variant"] == "CDiffE" and c["ydim"] > 24 and c["xdim"] <= 40 for c in ffma)
    assert {len(c["hidden"]) + 1 for c in ffma} >= {3, 5, 8}
    assert max(max(c["hidden"]) for c in ffma) >= 129 and min(min(c["hidden"]) for c in ffma) == 1
    assert any(c["variant"] == "DPS" and c["xdim"] == 128 for c in ffma)
    assert max(c["ydim"] for c in tc if c["variant"] == "CDE") == 300
    assert {c["l0_split"] for c in tc if c["inst"][2] is False and c["variant"] == "CDE"} == {1, 2, 3}
    fw = FORWARD_SWEEP.values()
    assert {2, 64, 65, 128, 129, 256, 512} <= {c["in_dim"] for c in fw if c["inst"] == FORWARD_INST}
    assert {1, 15, 17, 64, 127, 128} <= {c["out_dim"] for c in fw if c["inst"] == FORWARD_INST}
    assert {1, 30} <= {c["scale"] for c in fw if c["inst"] == FORWARD_INST}
    assert {129, 300} <= {c["out_dim"] for c in fw if c["inst"] == FFMA}


def test_every_sampler_group_has_a_guarded_case():
    assert {c["group"] for c in ALL_SAMPLER.values() if c.get("guard")} == {"A", "B", "C", "D", "E", "G"}


# ------------------------------------------------------------------------------------------- tests: the sweep can fail
# one representative case per group; each bug must move the checked rows by >= 5x the bf16 bound
MUTATION_CASES = {"A": "A-cde33+1", "B": "B-dps8+23", "C": "C-cdiffe9+24-split4-gain2", "D": "D-dps5+23-split4",
                  "E": "E-cde105+3", "G": "G-cde64+3-philox"}
SEPARATION = 5.0


def _mutation_rows(c, n_obs, n):
    rows = gc.sweep_rows(n_obs, n, 32 if c["group"] != "B" else K_TILE_M, seed=c["seed"])
    return rows if len(rows) <= 48 else np.concatenate([rows[:24], rows[-24:]])


@pytest.mark.parametrize("group", sorted(MUTATION_CASES))
def test_injected_sampler_bugs_miss_the_bf16_bound(group):
    c = ALL_SAMPLER[MUTATION_CASES[group]]
    n_obs, n = _runs(c)[-1]
    pb = gc.sampler_problem(c, n_obs, n)
    rows = _mutation_rows(c, n_obs, n)
    ref = gc.sampler_oracle(c, pb, rows)
    full = gc.sampler_oracle(c, pb, gc.sweep_rows(n_obs, n, 32 if c["group"] != "B" else K_TILE_M, seed=c["seed"],
                                                  n_random=16 if c["group"] != "B" else 64))
    tol = gc.SWEEP_TOL["sampler"]["bf16"] * full.abs().max().item()     # the scale the GPU case uses
    sep = {}
    for mut in gc.SAMPLER_MUTATIONS:
        if mut == "ynoise_previous" and c["variant"] != "CDiffE":
            continue
        sep[mut] = (gc.sampler_oracle(c, pb, rows, mut) - ref).abs().max().item() / tol
    assert min(sep.values()) >= SEPARATION, sep


def test_injected_forward_bugs_miss_the_bf16_bound():
    c = FORWARD_SWEEP["F-129to127-x1"]
    params, x, cond, t = gc.forward_problem(c, 300)
    ref = gc.forward_oracle(params, x, cond, t)
    scale = max(gc.forward_oracle(*gc.forward_problem(c, n)).abs().max().item() for n in c["ns"])
    tol = gc.SWEEP_TOL["forward"]["bf16"] * scale                       # the scale the GPU case uses
    sep = {mut: (gc.forward_oracle(params, x, cond, t, mut) - ref).abs().max().item() / tol
           for mut in gc.FORWARD_MUTATIONS}
    assert min(sep.values()) >= SEPARATION, sep


def _forward_bf16_emulated(params, inp):
    """the rounding the l0_split-4 forward is built with: f16 layer-0 operands, bf16 weights and activations in the
    hidden and output layers, fp32 accumulation"""
    W, b = params[0]
    h = torch.tanh(torch.tanh(inp.half().float() @ W.half().float().T + b))
    for W, b in params[1:-1]:
        h = torch.tanh(h.bfloat16().float() @ W.bfloat16().float().T + b)
    W, b = params[-1]
    return h.bfloat16().float() @ W.bfloat16().float().T + b


@pytest.mark.parametrize("name", sorted(n for n, c in FORWARD_SWEEP.items() if c["inst"] == FORWARD_INST
                                        and c["l0_split"] == 4))
def test_forward_cases_meet_the_bound_under_the_kernels_rounding(name):
    """each tensor-core forward case is one whose bound the kernel's designed arithmetic can meet, with the same
    normaliser as the GPU case: a miss on the GPU is then the kernel's, not the bound's"""
    c = FORWARD_SWEEP[name]
    err, scale = 0.0, 0.0
    for n in c["ns"]:
        if n == "multi":
            continue
        params, x, cond, t = gc.forward_problem(c, n)
        ref = gc.forward_oracle(params, x, cond, t)
        inp = torch.cat([x, t] if c["cls"] == "MLP2" else [x, cond, t], 1)
        err = max(err, (_forward_bf16_emulated(params, inp).double() - ref).abs().max().item())
        scale = max(scale, ref.abs().max().item())
    assert err <= 0.9 * gc.SWEEP_TOL["forward"]["bf16"] * scale, err / scale


# ------------------------------------------------------------------------------------------- tests: packing limits
@pytest.fixture(scope="module")
def lib():
    import dmip
    if not os.path.exists(dmip.library_path()):
        dmip.build()
    return dmip._lib.lib()


def _h3_desc(in_dim, out_dim):
    from dmip import _lib
    d = _lib.DmipMlp()
    d.n_layers, d.in_dim, d.out_dim = 4, in_dim, out_dim
    for i, w in enumerate(H3 + (out_dim,)):
        d.width[i] = w
    return d


@pytest.mark.parametrize("split,deepest", [(1, 512), (2, 256), (3, 168), (4, 512)])
def test_pack_bytes_refuses_a_layer0_depth_above_512(lib, split, deepest):
    """dmip_pack_bytes returns 0 (DMIP_EINVAL from tc_net_geom) one column past each l0_split's depth limit"""
    d = _h3_desc(600, 7)
    assert lib.dmip_pack_bytes(C.byref(d), deepest, 7, split) > 0
    assert lib.dmip_pack_bytes(C.byref(d), deepest + 1, 7, split) == 0
    assert b"exceeds 512" in lib.dmip_last_error()
    assert k0pad(deepest, split) <= 512 < k0pad(deepest + 1, split)


def test_pack_bytes_refuses_l0_split_5_and_wide_outputs(lib):
    d = _h3_desc(30, 7)
    assert lib.dmip_pack_bytes(C.byref(d), 29, 7, 4) > 0
    assert lib.dmip_pack_bytes(C.byref(d), 29, 7, 5) == 0
    assert b"l0_split" in lib.dmip_last_error()
    assert lib.dmip_pack_bytes(C.byref(_h3_desc(30, 129)), 29, 129, 4) == 0


def test_the_header_states_the_sampler_limits():
    src = open(os.path.join(ROOT, "include", "dmip.h")).read()
    for text in ("CDE xdim <= 104", "CDiffE xdim <= 32 and ydim <= 24", "DPS xdim <= 8", "[512,512,512]",
                 "DPS xdim <= 128"):
        assert text in src, text
