"""Throughput of the MMD permutation test (csrc/dmip_mmd_test.cu) on the GPU; writes ONE JSON line (default
profiles/mmd_test_bench.json).

    python tools/mmd_test_bench.py [--out FILE] [--skip-baselines]

Shapes: d = 3, one bandwidth, P = 254 permutations, n = m = 2^16 and 2^17, and the evaluate shape of 100 observations x
5000 x 5000.  For each: the kernel time of one dmip_mmd_test call (CUDA events, windows >= 1 s after a warm-up; the labels
are drawn once outside the timed window), the MUFU ceiling (N^2 ex2 at 16 lanes/clk/SM and the SM clock sampled during
the run) and the tensor ceiling (2 N^2 x 128 x 256 u8 operations: 128 bytes (hi, lo) per 64 points, nc = 256 accumulator
columns, at the data-sheet 4.5 POPS dense INT8 — the same time as 2 N^2 x 256 FLOP at 2.25 PFLOP/s f16), and which binds.  Baselines in the same run: (a) P + 1 dmip_mmd calls on the relabeled sets (timed on a
slice of the calls and scaled), (b) torch fp32 chunked cdist -> exp -> matmul with the 0/1 label matrix, TF32 off
(timed on a slice of the rows and scaled).  The line records the card name, power.limit and clocks.max.sm."""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.mmd_bench import EX2_PER_CLK, SMS, ClockSampler, smi, time_call  # noqa: E402

F16_DENSE_FLOPS = 2.25e15          # HGX B200 data sheet, dense FP16 / BF16 per GPU; dense INT8 is twice this


def relabeled_mmd_calls(x, y, first, sig, n_calls):
    """Baseline (a): dmip_mmd on the relabeled sets of the first n_calls permutations of observation 0."""
    from dmip import metrics
    z = torch.cat([x[0], y[0]])
    sets = [(z[f], z[~f]) for f in first[:n_calls]]

    def run():
        for a, b in sets:
            metrics.mmd2(a, b, sig)
    return run


def torch_matmul_baseline(x, y, sig, U, row_chunk, max_rows):
    """Baseline (b): rows of K in fp32 chunks, K_chunk @ U (N x nc 0/1 fp32), TF32 off; covers max_rows rows of obs 0."""
    z = torch.cat([x[0], y[0]])
    c = -1.0 / (2 * sig * sig)

    def run():
        acc = torch.zeros(U.shape[1], device=z.device)
        for r0 in range(0, max_rows, row_chunk):
            k = torch.cdist(z[r0:r0 + row_chunk], z).square_().mul_(c).exp_()
            acc += (k @ U).sum(0)
        return acc
    return run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "mmd_test_bench.json"))
    ap.add_argument("--skip-baselines", action="store_true")
    args = ap.parse_args()
    import dmip
    from dmip import metrics
    assert dmip.is_available(), "needs an sm_100 device and the built library (no fallback)"
    torch.cuda.set_device(0)
    torch.backends.cuda.matmul.allow_tf32 = False
    name, plimit, maxclk = (smi("name,power.limit,clocks.max.sm") or [torch.cuda.get_device_name(0), None, None])
    g = torch.Generator(device="cuda").manual_seed(0)
    P, sig = 254, [3 ** 0.5]
    cases = [("d3_n2^16_P254", 1, 1 << 16, 1 << 16), ("d3_n2^17_P254", 1, 1 << 17, 1 << 17),
             ("evaluate_100x5000x5000_d3_P254", 100, 5000, 5000)]
    res = {}
    with ClockSampler() as clk:
        for key, n_obs, n, m in cases:
            N = n + m
            x = torch.randn(n_obs, n, 3, device="cuda", generator=g)
            y = torch.randn(n_obs, m, 3, device="cuda", generator=g) * 1.1 + 0.05
            labels = metrics.permutation_labels(n_obs, n, m, P, generator=g)
            k0 = len(clk.samples)
            sec, reps, per = time_call(lambda: metrics.mmd2_permutation_statistics(x, y, sig, labels))
            mhz = float(np.mean(clk.samples[k0:])) if len(clk.samples) > k0 else None
            ex2 = n_obs * N * N * len(sig)                       # every (i, j) of the pooled matrix, every bandwidth
            flop = 2.0 * n_obs * N * N * 256
            entry = dict(n_obs=n_obs, n=n, m=m, d=3, n_bw=len(sig), n_perm=P, kernel_ms=sec * 1e3, calls_per_window=reps,
                         window_ms=[p * reps * 1e3 for p in per], sm_mhz=mhz,
                         tensor_ceiling_ms=flop / F16_DENSE_FLOPS * 1e3)
            if mhz:
                entry["mufu_ceiling_ms"] = ex2 / (SMS * EX2_PER_CLK * mhz * 1e6) * 1e3
                entry["binding_ceiling"] = "mufu" if entry["mufu_ceiling_ms"] > entry["tensor_ceiling_ms"] else "tensor"
                entry["fraction_of_binding_ceiling"] = max(entry["mufu_ceiling_ms"], entry["tensor_ceiling_ms"]) / (sec * 1e3)
            if not args.skip_baselines:
                first = torch.zeros(P + 1, N, dtype=torch.bool, device="cuda")
                first[0, :n] = True
                w = labels[0].to(torch.int64) & 0xffffffff
                bits = (w[:, :, None] >> torch.arange(32, device="cuda")) & 1
                first[1:] = bits.reshape(P, -1)[:, :N].bool()
                n_calls = 8
                s_a, _, _ = time_call(relabeled_mmd_calls(x, y, first, sig, n_calls), min_window=1.0, windows=1)
                entry["baseline_mmd_calls_ms"] = s_a / n_calls * (P + 1) * n_obs * 1e3
                U = torch.cat([first.T.float(), torch.ones(N, 1, device="cuda")], 1)
                rows = min(N, 4096)
                s_b, _, _ = time_call(torch_matmul_baseline(x, y, sig[0], U, 1024, rows), min_window=1.0, windows=1)
                entry["baseline_torch_cdist_exp_matmul_ms"] = s_b * (N / rows) * n_obs * 1e3
                entry["speedup_vs_mmd_calls"] = entry["baseline_mmd_calls_ms"] / entry["kernel_ms"]
                entry["speedup_vs_torch"] = entry["baseline_torch_cdist_exp_matmul_ms"] / entry["kernel_ms"]
            res[key] = entry
            print(key, json.dumps(entry), file=sys.stderr)
            del x, y, labels
            torch.cuda.empty_cache()
    line = dict(bench="mmd_test", card=name, power_limit_w=plimit, clocks_max_sm_mhz=maxclk,
                mufu_ex2_lanes_per_clk_per_sm_assumed=EX2_PER_CLK, f16_dense_flops_datasheet=F16_DENSE_FLOPS, cases=res)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(line) + "\n")
    print(json.dumps(line))


if __name__ == "__main__":
    main()
