"""Throughput of the kernel Stein discrepancy kernel (csrc/dmip_ksd.cu) on the GPU; writes ONE JSON line (default
profiles/ksd_bench.json).

    python tools/ksd_bench.py [--out FILE] [--ab-lib PARENT.so] [--tables]

For each case: kernel time from CUDA events over windows of >= 1 s after a warm-up, pair-scale evaluations/s (the kernel
evaluates n(n+1)/2 pairs per observation and scale: the tiles I <= J) and that rate over the ceiling of the kernel
instantiation the case runs, with the SM clock sampled during the run:
  - issue: 4 warp instructions per clock and SM (128 thread instructions) over the instructions per pair-scale of the
    inner column loop, counted in its SASS (`cuobjdump -sass`, DESIGN.md §3 "Evaluation metrics");
  - MUFU: 16 MUFU.RSQ / MUFU.EX2 lanes per clock and SM, one per pair-scale;
the smaller of the two binds.  Beside it a chunked fp32 torch baseline of the same Stein kernel timed on a slice of the
rows.  The line records the card name, power.limit, clocks.max.sm and the sampled SM clock.  --ab-lib loads another
build of the library beside this one and compares dmip_mmd's outputs bit for bit on the same inputs (and times both).
--tables adds the evaluate tables' KSD columns (reported, not gated): the trained linear CDE with the bf16 and fp32
samplers against exact posterior samples, and the scatterometry golden Metropolis and model sample sets."""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.mmd_bench import ClockSampler, smi, time_call  # noqa: E402
from tools import mmd_bench  # noqa: E402

SMS, ISSUE_PER_CLK, MUFU_PER_CLK = 148, 128, 16
# SASS instructions per pair-scale of the inner column loop, k_ksd<GAUSS, DP, NS, RPT> of this build: all instructions
# of the loop body over its MUFU count (one MUFU per pair and scale)
INSTR_PER_PAIR = {("imq", 2, 1): 914 / 88, ("gaussian", 2, 1): 834 / 88, ("imq", 3, 1): 1147 / 88,
                  ("gaussian", 3, 1): 709 / 56, ("imq", 3, 4): 615 / 88, ("gaussian", 3, 4): 572 / 88}


def bind(path):
    from dmip import metrics
    L = C.CDLL(path)
    L.dmip_ksd_workspace_bytes.restype = C.c_size_t
    L.dmip_ksd_workspace_bytes.argtypes = [C.POINTER(metrics.DmipKsd)]
    L.dmip_ksd.restype = C.c_int
    L.dmip_ksd.argtypes = [C.POINTER(metrics.DmipKsd), C.c_void_p]
    L.dmip_last_error.restype = C.c_char_p
    return L


def make_call(L, x, s, scales, kernel):
    """A closure that enqueues one dmip_ksd call on (n_obs, n, d) tensors; returns the output tensor."""
    from dmip import metrics
    n_obs, n, dim = x.shape
    d = metrics.DmipKsd()
    d.dim, d.n_obs, d.n, d.kernel, d.n_scales = dim, n_obs, n, metrics.KSD_KERNELS[kernel], len(scales)
    for i, c in enumerate(scales):
        d.scale[i] = c
    out = torch.empty(n_obs, len(scales), 2, dtype=torch.float64, device=x.device)
    nbytes = L.dmip_ksd_workspace_bytes(C.byref(d))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    d.x, d.score, d.out, d.workspace, d.workspace_bytes = x.data_ptr(), s.data_ptr(), out.data_ptr(), ws.data_ptr(), nbytes
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call():
        rc = L.dmip_ksd(C.byref(d), stream)
        if rc:
            raise RuntimeError(L.dmip_last_error().decode())
        return out
    call.keep = (x, s, out, ws, d)
    return call


def torch_baseline(x, s, scale, kernel, max_rows=4096):
    """Chunked fp32 torch evaluation of the Stein kernel sum (direct differences) on the first max_rows rows of each
    observation against all its columns; seconds per pair."""
    dim = x.shape[-1]
    row_chunk = max(1, min(max_rows, (1 << 26) // x.shape[1]))     # bounds the (rows, n, d) temporaries

    def run():
        tot = torch.zeros((), dtype=torch.float64, device=x.device)
        for o in range(x.shape[0]):
            xo, so = x[o], s[o]
            for r0 in range(0, min(xo.shape[0], max_rows), row_chunk):
                xa, sa = xo[r0:r0 + row_chunk], so[r0:r0 + row_chunk]
                delta = xa[:, None, :] - xo[None, :, :]
                r2 = delta.square().sum(-1)
                ss = sa @ so.T
                a = ((sa[:, None, :] - so[None, :, :]) * delta).sum(-1) + dim
                if kernel == "imq":
                    k = torch.rsqrt(r2 + scale * scale)
                    u = k * ss + k ** 3 * a - 3 * r2 * k ** 5
                else:
                    u = torch.exp(-r2 / (2 * scale * scale)) * (ss + a / scale ** 2 - r2 / scale ** 4)
                tot += u.sum(dtype=torch.float64)
        return tot
    sec, _, _ = time_call(run, windows=1)
    rows = min(x.shape[1], max_rows)
    return sec / (x.shape[0] * rows * x.shape[1])


def ab_mmd(L_ab_path, g):
    """dmip_mmd of this build against another build on the same inputs: bit equality of every output, and times."""
    import dmip
    La, Lb = mmd_bench.bind(dmip.library_path()), mmd_bench.bind(os.path.abspath(L_ab_path))
    res = {}
    for key, n_obs, n, m, d, sig in [("d3_2^18_bw1", 1, 1 << 18, 1 << 18, 3, [1.0]), ("d1_3x129x4099_bw8", 3, 129, 4099, 1,
                                     [0.2, 0.3, 0.5, 0.7, 1.0, 1.5, 2.0, 3.0]), ("d5_5x1000x777_bw3", 5, 1000, 777, 5,
                                     [0.5, 1.0, 2.0]), ("d16_2x2049x515_bw2", 2, 2049, 515, 16, [2.0, 4.0]),
                                    ("evaluate_100x5000x5000_d3_bw1", 100, 5000, 5000, 3, [1.0])]:
        x = torch.randn(n_obs, n, d, device="cuda", generator=g)
        y = torch.randn(n_obs, m, d, device="cuda", generator=g) * 1.1 + 0.05
        fa, fb = mmd_bench.make_call(La, x, y, sig), mmd_bench.make_call(Lb, x, y, sig)
        a, b = fa().clone(), fb().clone()
        torch.cuda.synchronize()
        res[key] = dict(bit_identical=bool(torch.equal(a.view(torch.int64), b.view(torch.int64))),
                        max_abs_diff=float((a - b).abs().max()))
        if key.startswith("d3_2^18") or key.startswith("evaluate"):
            ta, tb = [], []
            for _ in range(3):
                ta.append(time_call(fa, windows=1)[0])
                tb.append(time_call(fb, windows=1)[0])
            res[key].update(this_build_ms=[t * 1e3 for t in ta], other_build_ms=[t * 1e3 for t in tb],
                            other_over_this=float(np.median(tb) / np.median(ta)))
        print("ab_mmd", key, json.dumps(res[key]), file=sys.stderr)
    return dict(other_lib=os.path.basename(L_ab_path), cases=res)


def tables():
    """KSD columns of the evaluate tables: IMQ KSD^2_U summed over the scales, mean over repeats, per observation."""
    import gpu_cases as gc
    from util import load_golden
    from dmip import evaluation
    from dmip.linear_problem import LinearForwardProblem
    from dmip.models.diffusion import CDE
    from dmip.utils_scatterometry import make_score_posterior
    from oracle.weights import make_params, state_dict_from_params
    out = {}
    z = np.load(os.path.join(ROOT, "tests", "golden", "trained_cde_linear.npz"))
    model = CDE(2, 2, [512, 512, 512])
    model.sde.a.load_state_dict({f"{k}.{p}": torch.from_numpy(z[f"{k}_{p}"]) for k in (0, 3, 5, 7)
                                 for p in ("weight", "bias")})
    model.sde.to("cuda")
    ys = load_golden("eval_linear", dtype=torch.float64)["ys"].float()
    sc = (0.25, 0.5, 1.0)
    for prec in ("fp32", "bf16"):
        model.precision = prec
        torch.manual_seed(0)
        _, _, _, t = evaluation.evaluate_linear(model, ys, LinearForwardProblem(), n_samples_x=5000, n_repeats=10,
                                                ksd_scales=sc)
        out[f"linear_trained_cde_{prec}"] = dict(ys=ys.tolist(), n=5000, repeats=10, ksd_scales=sc,
                                                 **{k: np.asarray(v).tolist() for k, v in t.items()})
    fx = load_golden("eval_scat", dtype=torch.float64)
    xp, xt = fx["x_pred"].float(), fx["x_true"].float()
    fm, _ = gc._surrogate_module()
    m = CDE(3, 23, [512, 512, 512])
    m.sde.a.load_state_dict(state_dict_from_params(make_params(95, 27, 3)))
    m.sde.to("cuda")
    m.sde.a.precision = "fp32"
    sp = make_score_posterior(fm, dict(a=0.2, b=0.01, lambd_bd=1000))
    sets = lambda v: [v[:, j].contiguous().cuda() for j in range(v.shape[1])]
    sc = (0.1, 0.3, 1.0)
    t = evaluation.scatterometry_metrics(m, fx["ys"].float(), fm, sets(xp), sets(xt), sp, 0.2, 0.01, 1000, ksd_scales=sc)
    out["scatterometry_golden_sets"] = dict(n=int(xp.shape[2]), repeats=int(xp.shape[1]), ksd_scales=sc,
                                            **{k: np.asarray(v).tolist() for k, v in t.items()})
    for k, v in out.items():
        print("tables", k, json.dumps(v), file=sys.stderr)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ksd_bench.json"))
    ap.add_argument("--ab-lib", default=None)
    ap.add_argument("--tables", action="store_true")
    args = ap.parse_args()
    import dmip
    assert dmip.is_available(), "needs an sm_100 device and the built library (no fallback)"
    torch.cuda.set_device(0)
    name, plimit, maxclk = (smi("name,power.limit,clocks.max.sm") or [torch.cuda.get_device_name(0), None, None])
    L = bind(dmip.library_path())
    g = torch.Generator(device="cuda").manual_seed(0)
    N = 1 << 20
    cases = [("imq_d2_n2^20_c1", "imq", 1, N, 2, [1.0]), ("gaussian_d2_n2^20_s1", "gaussian", 1, N, 2, [1.0]),
             ("imq_d3_n2^20_c1", "imq", 1, N, 3, [1.0]), ("gaussian_d3_n2^20_s1", "gaussian", 1, N, 3, [1.0]),
             ("imq_d3_n2^20_c4", "imq", 1, N, 3, [0.25, 0.5, 1.0, 2.0]),
             ("gaussian_d3_n2^20_s4", "gaussian", 1, N, 3, [0.25, 0.5, 1.0, 2.0]),
             ("imq_evaluate_100x5000_d3_c1", "imq", 100, 5000, 3, [1.0]),
             ("gaussian_evaluate_100x5000_d3_s1", "gaussian", 100, 5000, 3, [1.0])]
    res = {}
    with ClockSampler() as clk:
        for key, kernel, n_obs, n, d, sc in cases:
            x = torch.randn(n_obs, n, d, device="cuda", generator=g) * 0.8 + 0.1
            s = -1.3 * x + 0.2 * torch.randn(n_obs, n, d, device="cuda", generator=g)
            k0 = len(clk.samples)
            sec, reps, per = time_call(make_call(L, x, s, sc, kernel))
            mhz = float(np.mean(clk.samples[k0:])) if len(clk.samples) > k0 else None
            ev = n_obs * len(sc) * n * (n + 1) / 2
            ipp = INSTR_PER_PAIR[(kernel, d, len(sc))]
            entry = dict(kernel=kernel, n_obs=n_obs, n=n, d=d, n_scales=len(sc), kernel_ms=sec * 1e3,
                         calls_per_window=reps, window_ms=[p * reps * 1e3 for p in per], pair_scale_evals_per_s=ev / sec,
                         sm_mhz=mhz, sass_instr_per_pair_scale=ipp)
            if mhz:
                issue = SMS * ISSUE_PER_CLK / ipp * mhz * 1e6
                mufu = SMS * MUFU_PER_CLK * mhz * 1e6
                entry.update(issue_ceiling_per_s=issue, mufu_ceiling_per_s=mufu,
                             binding="issue" if issue < mufu else "mufu",
                             fraction_of_ceiling=ev / sec / min(issue, mufu))
            spp = torch_baseline(x, s, sc[0], kernel)
            entry["torch_fp32_pair_evals_per_s"] = 1.0 / spp
            entry["speedup_vs_torch_per_scale"] = ev / sec / len(sc) * spp
            res[key] = entry
            print(key, json.dumps(entry), file=sys.stderr)
            del x, s
            torch.cuda.empty_cache()
        if args.ab_lib:
            res["ab_mmd"] = ab_mmd(args.ab_lib, g)
        all_mhz = list(clk.samples)
    if args.tables:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        res["evaluate_tables"] = tables()
    line = dict(bench="ksd", card=name, power_limit_w=plimit, clocks_max_sm_mhz=maxclk,
                sm_mhz_sampled_mean=float(np.mean(all_mhz)) if all_mhz else None,
                sm_mhz_sampled_min=float(np.min(all_mhz)) if all_mhz else None, cases=res)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(line) + "\n")
    print(json.dumps(line))


if __name__ == "__main__":
    main()
