"""The fused samplers and the score-net forward at every kernel instantiation, state width and tile tail, against the
fp64 oracle (pytest -m gpu).  The cases and the dispatch table they are checked against are in
tests/test_sampler_sweep_plan.py:
  A  CDE on tcgen05: xdim 1 ... 104 (NP 1 / 4 / 13), both layer-0 operand locations, ydim 1 ... 300;
  B  persistent tiles: more tiles than two rounds of the grid, tcgen05 against FFMA on all rows;
  C  CDiffE on tcgen05: (xdim, ydim) up to (32, 24);
  D  DPS on tcgen05: xdim 1 ... 8, ydim up to 200;
  E  the FFMA sampler: net shapes and states past the tcgen05 limits (precision 'bf16' must fall back);
  F  the forward on tcgen05 and FFMA: in_dim 2 ... 512, out_dim 1 ... 300, every l0_split at its depth limit;
  G  in-kernel Philox against its injected mirror, the VE-SDE with a corrector, at NP 4 and 13;
  H  descriptors outside the kernels' limits are refused at the C ABI.
Every call asserts the path that ran (`last_precision`), so a tensor-core case cannot pass on the FFMA kernels.
One case per sampler group runs under DMIP_GUARD=1 (canaries around the sampler's output)."""
import pytest

import gpu_cases as gc
import test_sampler_sweep_plan as plan

pytestmark = pytest.mark.gpu

RATIOS = {}      # group -> worst err / tol seen in this session (printed at the end of the module)


@pytest.fixture(scope="module", autouse=True)
def _report(request):
    yield
    tr = request.config.pluginmanager.get_plugin("terminalreporter")
    if tr is not None and RATIOS:
        tr.write_line("")
        for g in sorted(RATIOS):
            tr.write_line(f"sampler sweep: group {g}: worst err/tol {RATIOS[g][0]:.3f} ({RATIOS[g][1]})")


def _ok(group, name, res):
    err, tol, detail = res
    if err <= tol and err / tol >= RATIOS.get(group, (-1.0, ""))[0]:
        RATIOS[group] = (err / tol, name)
    assert err <= tol, (name, err, tol, detail)


@pytest.fixture
def guard(monkeypatch):
    def on(c):
        if c.get("guard"):
            monkeypatch.setenv("DMIP_GUARD", "1")
    return on


@pytest.mark.parametrize("name", sorted(plan.SAMPLER_SWEEP))
def test_sampler_sweep(name, guard):
    c = plan.SAMPLER_SWEEP[name]
    guard(c)
    _ok(c["group"], name, gc.case_sampler_sweep(c, plan.sampler_paths(c)))


@pytest.mark.parametrize("name", sorted(plan.PERSISTENT))
def test_sampler_persistent_tiles(name, guard):
    c = plan.PERSISTENT[name]
    guard(c)
    _ok("B", name, gc.case_sampler_persistent(c))


@pytest.mark.parametrize("name", sorted(plan.FORWARD_SWEEP))
def test_forward_sweep(name):
    c = plan.FORWARD_SWEEP[name]
    _ok("F", name, gc.case_forward_sweep(c, plan.forward_paths(c)))


@pytest.mark.parametrize("name", sorted(plan.ABI_REJECTED))
def test_the_c_abi_refuses_shapes_past_the_limits(name):
    from dmip import _lib
    desc, match = plan.ABI_REJECTED[name]
    desc = dict(desc, variant={"CDE": _lib.CDE, "CDiffE": _lib.CDIFFE, "DPS": _lib.DPS}[desc["variant"]],
                precision=_lib.precision_code(desc["precision"]))
    err, tol, detail = gc.case_sampler_abi_rejects(desc, match)
    assert err <= tol, (name, detail)
