"""Throughput of the MMD^2 kernel (csrc/dmip_mmd.cu) on the GPU; writes ONE JSON line (default profiles/mmd_bench.json).

    python tools/mmd_bench.py [--out FILE] [--ab-lib OTHER.so] [--no-parity]

For each case: kernel time from CUDA events over windows of >= 1 s after a warm-up, pair-bandwidth evaluations/s
(the kernel evaluates n(n-1)/2 + m(m-1)/2 + n m pairs per observation and bandwidth: the XX / YY terms by symmetry) and
that rate over the MUFU ceiling 148 SMs x 16 ex2/clk x the SM clock sampled during the run.  Beside it a chunked fp32
torch baseline (cdist -> exp -> sum) on the same shape, timed on a slice of the rows.  The line records the card name,
power.limit, clocks.max.sm and the sampled SM clock.  --ab-lib alternates the product library with another build of it
on the d = 3 headline case and checks both against float64.  Unless --no-parity it also
reports (no threshold) MMD^2_u between bf16 and fp32 samples of the trained linear CDE at 2^20 particles, with two
independent fp32 runs beside it."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SMS, EX2_PER_CLK = 148, 16


def smi(fields):
    try:
        r = subprocess.run(["nvidia-smi", f"--query-gpu={fields}", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return [v.strip() for v in r.stdout.strip().splitlines()[0].split(",")]
    except Exception:
        return None


class ClockSampler:
    """Samples clocks.sm every 100 ms in a thread while timed windows run."""

    def __init__(self):
        self.samples, self.on, self.t = [], False, None

    def _run(self):
        while self.on:
            v = smi("clocks.sm")
            if v:
                try:
                    self.samples.append(float(v[0]))
                except ValueError:
                    pass
            time.sleep(0.1)

    def __enter__(self):
        self.on = True
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()
        return self

    def __exit__(self, *a):
        self.on = False
        self.t.join()


def bind(path):
    from dmip import metrics
    L = C.CDLL(path)
    L.dmip_mmd_workspace_bytes.restype = C.c_size_t
    L.dmip_mmd_workspace_bytes.argtypes = [C.POINTER(metrics.DmipMmd)]
    L.dmip_mmd.restype = C.c_int
    L.dmip_mmd.argtypes = [C.POINTER(metrics.DmipMmd), C.c_void_p]
    L.dmip_last_error.restype = C.c_char_p
    return L


def make_call(L, x, y, sigmas):
    """A closure that enqueues one dmip_mmd call on (n_obs, n, d) / (n_obs, m, d) tensors; returns the output tensor."""
    from dmip import metrics
    n_obs, n, dim = x.shape
    d = metrics.DmipMmd()
    d.dim, d.n_obs, d.n, d.m, d.n_bw = dim, n_obs, n, y.shape[1], len(sigmas)
    for i, s in enumerate(sigmas):
        d.sigma[i] = s
    out = torch.empty(n_obs, len(sigmas), 4, dtype=torch.float64, device=x.device)
    nbytes = L.dmip_mmd_workspace_bytes(C.byref(d))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    d.x, d.y, d.out, d.workspace, d.workspace_bytes = x.data_ptr(), y.data_ptr(), out.data_ptr(), ws.data_ptr(), nbytes
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call():
        rc = L.dmip_mmd(C.byref(d), stream)
        if rc:
            raise RuntimeError(L.dmip_last_error().decode())
        return out
    call.keep = (x, y, out, ws, d)
    return call


def time_call(fn, min_window=1.0, windows=3):
    """Median seconds per call over `windows` event-timed windows of >= min_window s each (after one warm-up call)."""
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    reps = max(1, int(np.ceil(min_window / max(time.perf_counter() - t0, 1e-6))))
    per = []
    for _ in range(windows):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        b.synchronize()
        per.append(a.elapsed_time(b) / 1e3 / reps)
    return float(np.median(per)), reps, per


def pair_evals(n_obs, n, m, nb):
    return n_obs * nb * (n * (n - 1) / 2 + m * (m - 1) / 2 + n * m)


def torch_baseline(x, y, sigma, row_chunk=1024, max_rows=8192):
    """Chunked fp32 cdist -> exp -> sum on the first max_rows rows of each term; seconds per pair."""
    c = -1.0 / (2 * sigma * sigma)

    def run():
        tot = torch.zeros((), dtype=torch.float64, device=x.device)
        for o in range(x.shape[0]):
            for a, b in ((x[o], x[o]), (y[o], y[o]), (x[o], y[o])):
                for r0 in range(0, min(a.shape[0], max_rows), row_chunk):
                    d2 = torch.cdist(a[r0:r0 + row_chunk], b).square_()
                    tot += d2.mul_(c).exp_().sum(dtype=torch.float64)
        return tot
    sec, reps, _ = time_call(run)
    rows = min(x.shape[1], max_rows)
    pairs = x.shape[0] * (rows * x.shape[1] + min(y.shape[1], max_rows) * y.shape[1] + rows * y.shape[1])
    return sec / pairs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "mmd_bench.json"))
    ap.add_argument("--ab-lib", default=None)
    ap.add_argument("--ab-rounds", type=int, default=3)
    ap.add_argument("--no-parity", action="store_true")
    args = ap.parse_args()
    import dmip
    from dmip import metrics
    from oracle import mmd as om
    assert dmip.is_available(), "needs an sm_100 device and the built library (no fallback)"
    torch.cuda.set_device(0)
    name, plimit, maxclk = (smi("name,power.limit,clocks.max.sm") or [torch.cuda.get_device_name(0), None, None])
    L = bind(dmip.library_path())
    g = torch.Generator(device="cuda").manual_seed(0)
    N = 1 << 20
    cases = [("d2_n2^20_bw1", 1, N, N, 2, [1.0]), ("d3_n2^20_bw1", 1, N, N, 3, [1.0]),
             ("d3_n2^20_bw4", 1, N, N, 3, [0.25, 0.5, 1.0, 2.0]), ("evaluate_100x5000x5000_d3_bw1", 100, 5000, 5000, 3, [1.0]),
             ("ex2_probe_d1_n2^18_bw8", 1, 1 << 18, 1 << 18, 1, [0.5, 0.6, 0.7, 0.8, 0.9, 1.0, 1.1, 1.2])]
    res = {}
    with ClockSampler() as clk:
        for key, n_obs, n, m, d, sig in cases:
            x = torch.randn(n_obs, n, d, device="cuda", generator=g)
            y = torch.randn(n_obs, m, d, device="cuda", generator=g) * 1.1 + 0.05
            k0 = len(clk.samples)
            sec, reps, per = time_call(make_call(L, x, y, sig))
            mhz = float(np.mean(clk.samples[k0:])) if len(clk.samples) > k0 else None
            ev = pair_evals(n_obs, n, m, len(sig))
            entry = dict(n_obs=n_obs, n=n, m=m, d=d, n_bw=len(sig), kernel_ms=sec * 1e3, calls_per_window=reps,
                         window_ms=[p * reps * 1e3 for p in per], pair_bw_evals_per_s=ev / sec, sm_mhz=mhz)
            if mhz:
                entry["mufu_ceiling_per_s"] = SMS * EX2_PER_CLK * mhz * 1e6
                entry["fraction_of_mufu_ceiling"] = ev / sec / entry["mufu_ceiling_per_s"]
            if not key.startswith("ex2_probe"):
                spp = torch_baseline(x, y, sig[0])
                entry["torch_fp32_pair_evals_per_s"] = 1.0 / spp          # one bandwidth
                entry["speedup_vs_torch_per_bandwidth"] = ev / sec / len(sig) * spp
            res[key] = entry
            print(key, json.dumps(entry), file=sys.stderr)
            del x, y
            torch.cuda.empty_cache()
        if args.ab_lib:
            La = bind(os.path.abspath(args.ab_lib))
            x = torch.randn(1, N, 3, device="cuda", generator=g)
            y = torch.randn(1, N, 3, device="cuda", generator=g) * 1.1 + 0.05
            fa, fb = make_call(L, x, y, [1.0]), make_call(La, x, y, [1.0])
            ta, tb = [], []
            for _ in range(args.ab_rounds):
                ta.append(time_call(fa, windows=1)[0])
                tb.append(time_call(fb, windows=1)[0])
            # accuracy of both builds against float64 on a size the oracle handles
            xs = torch.randn(2, 3000, 3, generator=torch.Generator().manual_seed(5))
            ys = torch.randn(2, 2500, 3, generator=torch.Generator().manual_seed(6)) * 1.2 + 0.3
            sig = [0.3, 1.0, 3.0]
            ref = np.stack([om.mmd2_terms(xs[o].numpy(), ys[o].numpy(), sig) for o in range(2)])
            err = {}
            for tag, LL in (("product", L), ("ab_lib", La)):
                got = make_call(LL, xs.cuda(), ys.cuda(), sig)().cpu().numpy()
                err[tag] = dict(terms=float(np.abs(got[..., 1:] - ref[..., 1:]).max()),
                                mmd=float(np.abs(got[..., 0] - ref[..., 0]).max()))
            res["ab"] = dict(lib=os.path.basename(args.ab_lib), product_ms=[t * 1e3 for t in ta],
                             ab_lib_ms=[t * 1e3 for t in tb], ab_over_product=float(np.median(tb) / np.median(ta)),
                             max_abs_err_vs_float64=err)
            print("ab", json.dumps(res["ab"]), file=sys.stderr)
        all_mhz = list(clk.samples)
    if not args.no_parity:
        from dmip.models.diffusion import CDE
        z = np.load(os.path.join(ROOT, "tests", "golden", "trained_cde_linear.npz"))
        model = CDE(2, 2, [512, 512, 512])
        model.sde.a.load_state_dict({f"{k}.{p}": torch.from_numpy(z[f"{k}_{p}"]) for k in (0, 3, 5, 7)
                                     for p in ("weight", "bias")})
        model.sde.to("cuda")
        yobs = torch.tensor([0.4, -0.7])
        draw = lambda prec, seed: model(yobs, num_samples=N, num_steps=200, precision=prec, seed=seed, return_tensor=True)
        f1, f2, b1 = draw("fp32", 1), draw("fp32", 2), draw("bf16", 3)
        bw = metrics.median_bandwidth(f1, f2)
        sig = [bw / 4, bw / 2, bw, 2 * bw]
        res["sampler_parity_trained_cde_linear"] = dict(
            particles=N, num_steps=200, y=[0.4, -0.7], median_bandwidth=bw, bandwidths=sig,
            mmd2_fp32_vs_bf16=metrics.mmd2(f1, b1, sig).tolist(), mmd2_fp32_vs_fp32=metrics.mmd2(f1, f2, sig).tolist())
    line = dict(bench="mmd", card=name, power_limit_w=plimit, clocks_max_sm_mhz=maxclk,
                sm_mhz_sampled_mean=float(np.mean(all_mhz)) if all_mhz else None,
                sm_mhz_sampled_min=float(np.min(all_mhz)) if all_mhz else None,
                mufu_ex2_lanes_per_clk_per_sm_assumed=EX2_PER_CLK, cases=res)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(line) + "\n")
    print(json.dumps(line))


if __name__ == "__main__":
    main()
