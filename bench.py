#!/usr/bin/env python
"""bench.py — headline benchmark of the dmip-b200 hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload ...] [--no-also]
                    [--dump-outputs DIR]

Headline workload (BASELINE.json configs[4], the config the metric "score-net evals/sec at 1/2/4/8 B200 + % tensor peak"
is quoted on): synthetic CDE score net, xdim 100, ydim 27 (SURVEY.md §8a), hidden [512,512,512], weights
torch.manual_seed(0) default init, one observation y ~ N(0,I) (seed 1), --particles (default 1,048,576) per GPU,
--sde-steps (default 1000) Euler–Maruyama steps, Philox seed 1234.  One bench "step" = one full posterior-sampling
call  model(y, num_samples=particles, num_steps=sde_steps)  = particles x sde_steps score-net evaluations = ONE launch
of the persistent kernel k_tc_mlp.  Weak scaling: every rank integrates its own `particles` (global particle index
offset = rank * particles; no communication on the hot loop).

`value`    — evals/s with y and the samples resident in HBM (CUDA events around the K calls, max over ranks).
`e2e`      — the same metric through the reference-facing call with HOST buffers: y is a pinned host tensor, the result
             is the numpy array the reference returns (device->host copy inside the timed region).
`roofline` — tensor bound: achieved = evals/s x F (F = algorithmic FLOP per evaluation, unpadded dims, tanh / SDE
             update not counted, SURVEY.md §8d) vs the measured SUSTAINED bf16 cuBLAS peak (the kernel runs > 1 s).
`cpu_baseline` / `--impl reference` — the reference's OWN classes (models/diffusion.py CDE.__call__, staged unmodified
             under baseline/_ref by baseline/make_ref.py) on the host cores, on a bounded sample of the same workload;
             the oracle port (oracle/sampler.py) only if the staged sources are missing — `kind` says which ran.
`also`     — the other BASELINE configs as short runs on the same JSON line, each with its own value / ms / roofline /
             e2e: cdiffe_scat = configs[2] (scatterometry CDiffE, 1M x 1000), dps_scat = configs[3] per-GPU share
             (32 observations x 65,536 particles), pinn_linear = configs[1] (linear CDE, PINNLoss fwd+bwd+Adam at batch
             65,536), dsm_linear (the DSM step at the same batch), posterior_loss (DPS joint loss, batch 16,384),
             surrogate_score (K4 at 256 x 65,536 rows), sweep (configs[4] at 64K ... 16M particles, S = 200);
             for --gpus N > 1: pinn_dp, the data-parallel PINN step (gradient all-reduce over NCCL) instead.
The same workloads can be run alone with --workload (then they are the JSON line's headline).

`--dump-outputs DIR` (sampler workloads) writes the samples the last timed call returned as DIR/samples.npy (float32,
rows = particles in global order, observation-major for dps_scat).  Above DUMP_ROWS rows it keeps a fixed sample of
DUMP_ROWS rows (seeded, sorted row indices), so the file stays small and two builds run with the same arguments can be
compared row for row: weights, observations and the Philox noise are seeded, so the inputs are identical from run to run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HIDDEN = [512, 512, 512]
WORKLOADS = {
    # name: (model class, xdim, ydim, n_obs per GPU, default particles per observation, default SDE steps)
    "synthetic": ("CDE", 100, 27, 1, 1 << 20, 1000),
    "cdiffe_scat": ("CDiffE", 3, 23, 1, 1 << 20, 1000),
    "dps_scat": ("Posterior", 3, 23, 32, 1 << 16, 1000),
}
SURR_FLOP = 2 * 2 * (3 * 256 + 256 * 256 * 2 + 256 * 23)       # surrogate forward + reverse sweep = 550,912 FLOP / row
DUMP_ROWS = 1 << 16          # --dump-outputs: 65,536 rows x at most 100 floats = at most 26 MB of samples


def flop_per_eval(kind, xdim, ydim):
    """Algorithmic FLOPs of one score evaluation (SURVEY.md §8: 2 (in 512 + 512 512 + 512 512 + 512 out))."""
    def net(i, o):
        return 2 * (i * 512 + 512 * 512 + 512 * 512 + 512 * o)
    if kind == "CDE":
        return net(xdim + ydim + 1, xdim)
    if kind == "CDiffE":
        return net(xdim + ydim + 1, xdim + ydim)
    return net(xdim + 1, xdim) + net(xdim + ydim + 1, xdim)      # DPS: prior + likelihood net


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--particles", type=int, default=0, help="particles per observation per GPU (0 = workload default)")
    ap.add_argument("--sde-steps", type=int, default=0)
    ap.add_argument("--precision", default="bf16")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="headline line only (skip the other BASELINE configs)")
    ap.add_argument("--workload", default="synthetic",
                    choices=list(WORKLOADS) + ["pinn_linear", "dsm_linear", "posterior_loss", "surrogate_score", "mcmc_scat"],
                    help="synthetic = BASELINE configs[4] (the headline line); the others are configs[2], [3], [1], ...")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the samples of the last timed call as DIR/samples.npy (sampler workloads)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload not in WORKLOADS):
        ap.error(f"--dump-outputs needs --impl ours and a sampler workload ({', '.join(WORKLOADS)})")
    return args


# ----------------------------------------------------------------------------------------------- stdout discipline
_REAL_STDOUT = None


def claim_stdout():
    """rank 0 prints ONE JSON line on stdout; everything else that writes to fd 1 (NCCL's INFO log, library banners) is
    sent to stderr instead — the log stays available to the driver without polluting the JSON."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
        sys.stdout = sys.stderr


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


# ----------------------------------------------------------------------------------------------- CPU baseline
def cpu_params(in_dim, out_dim, seed=0):
    """nn.Linear default init under torch.manual_seed(seed), built on CPU (the GPU arm's synthetic weights)."""
    import torch
    torch.manual_seed(seed)
    dims = [in_dim] + HIDDEN + [out_dim]
    layers = [torch.nn.Linear(a, b) for a, b in zip(dims[:-1], dims[1:])]
    return [(l.weight.detach().clone(), l.bias.detach().clone()) for l in layers]


_REF_MODEL = {}


def _reference_cde(xdim, ydim, cls="CDE"):
    """The stock reference class on CPU (baseline/_ref = unmodified reference files; oracle/shims for the three modules
    the reference tree does not contain).  None if the staged sources are missing.  For cls != 'CDE' the reference's
    losses module is attached as `model.ref_losses` (the training arm needs its DSMLoss)."""
    key = (xdim, ydim, cls)
    if key in _REF_MODEL:
        return _REF_MODEL[key]
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    model = None
    if os.path.exists(os.path.join(ref_dir, "models", "diffusion.py")):
        import importlib
        import torch
        saved_path, saved_mods = list(sys.path), {k: sys.modules.get(k) for k in ("models", "sdes", "nets", "losses")}
        avail = torch.cuda.is_available
        try:
            sys.path[:0] = [ref_dir, os.path.join(ROOT, "oracle", "shims")]
            for k in saved_mods:
                sys.modules.pop(k, None)
            torch.cuda.is_available = lambda: False        # the reference picks its device at import time: keep it on CPU
            mod = importlib.import_module("models.diffusion")
            torch.manual_seed(0)
            model = getattr(mod, cls)(xdim, ydim, list(HIDDEN))
            model.ref_losses = importlib.import_module("losses")
            if cls == "CDE":
                model.sde.eval()
        except Exception as e:                             # noqa: BLE001 — fall back to the port, and say so
            print("reference arm: stock classes unavailable:", repr(e), file=sys.stderr)
            model = None
        finally:
            torch.cuda.is_available = avail
            sys.path[:] = saved_path
            for k, v in saved_mods.items():
                sys.modules.pop(k, None)
                if v is not None:
                    sys.modules[k] = v
    _REF_MODEL[key] = model
    return model


def cpu_sampler_rate(n, s, xdim=100, ydim=27):
    """Time the reference sampler on n particles x s steps on all host cores.  Returns (evals/s, cores, seconds, kind):
    kind 'reference' = the stock CDE.__call__ of the reference (torch's own RNG, the per-step ones*ts[i] / cat / addmm
    of models/diffusion.py:27-46); kind 'port' = oracle/sampler.py, only when baseline/_ref is missing."""
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    g = torch.Generator().manual_seed(1)
    y = torch.randn(ydim, generator=g)
    model = _reference_cde(xdim, ydim)
    with torch.no_grad():
        if model is not None:
            model(y, num_samples=256, num_steps=2)                              # warm-up
            t0 = time.perf_counter()
            model(y, num_samples=n, num_steps=s)
            return n * s / (time.perf_counter() - t0), cores, time.perf_counter() - t0, "reference"
        from oracle import sampler as osamp            # fallback: the one other place bench.py may execute oracle/
        params = cpu_params(xdim + ydim + 1, xdim)
        x0 = torch.randn(n, xdim, generator=g)
        noise = torch.randn(1, n, xdim, generator=g).expand(s, n, xdim)   # one draw reused: timing is unaffected
        osamp.em_sampler_cde(params, y, x0[:256], noise[:2, :256], 2)
        t0 = time.perf_counter()
        osamp.em_sampler_cde(params, y, x0, noise, s)
        dt = time.perf_counter() - t0
    return n * s / dt, cores, dt, "port"


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        rows = [r for ts, r in self.rows if t0 <= ts <= t1 + 0.3 and len(r) >= 7] or [r for _, r in self.rows if len(r) >= 7]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = [float(r[0]) for r in rows if r[0].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": float(rows[0][1]), "reasons": reasons,
                "samples": len(rows)}


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def load_traffic():
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return {}


_FP32_PEAK = {}


def measured_fp32_tflops():
    """Denominator for the kernels that are fp32 FFMA by design (K4 surrogate, Metropolis): the cuBLAS SGEMM rate with
    TF32 off, measured live on this GPU (8192^3, best of 5) — a measured peak instead of the nominal 72 TFLOP/s."""
    import torch
    dev = torch.cuda.current_device()
    if dev not in _FP32_PEAK:
        old = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = False
        try:
            a = torch.randn(8192, 8192, device="cuda")
            b = torch.randn(8192, 8192, device="cuda")
            best = 1e9
            for i in range(6):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                torch.matmul(a, b)
                e1.record()
                torch.cuda.synchronize()
                if i:
                    best = min(best, e0.elapsed_time(e1))
            _FP32_PEAK[dev] = 2 * 8192 ** 3 / (best * 1e-3) / 1e12
        finally:
            torch.backends.cuda.matmul.allow_tf32 = old
        del a, b
    return _FP32_PEAK[dev]


def tensor_roofline(ach_tf, sustained, **extra):
    """roofline object against the measured bf16 tensor peak (MEASURED_PEAKS.json; fallback of B200_PROFILING.md)"""
    peaks = load_peaks()
    key = "bf16_tflops_sustained" if sustained else "bf16_tflops"
    peak = peaks.get(key)
    src = f"measured {'sustained' if sustained else 'burst'} bf16 cuBLAS (MEASURED_PEAKS.json)"
    if not peak:
        peak, src = (1400.0 if sustained else 1590.0), "fallback bf16 peak (B200_PROFILING.md)"
    r = {"bound": "tensor", "achieved": ach_tf, "peak": peak, "unit": "TFLOP/s", "frac": ach_tf / peak, "traffic": None,
         "peak_source": src}
    r.update(extra)
    return r


# ----------------------------------------------------------------------------------------------- reference arm
CFG_NAMES = {"synthetic": "configs[4]: synthetic CDE", "cdiffe_scat": "configs[2]: scatterometry CDiffE",
             "dps_scat": "configs[3] (per-GPU share): scatterometry DPS"}


def workload_name(args):
    """`config.workload` of the sampler workloads — the same string on our arm and on the reference arm"""
    kind, xdim, ydim, n_obs, n_def, s_def = WORKLOADS[args.workload]
    N, S = args.particles or n_def, args.sde_steps or s_def
    return (f"{CFG_NAMES[args.workload]} xdim={xdim} ydim={ydim} hidden=512x3, {n_obs} observation(s) x "
            f"{N} particles per GPU x {S} SDE steps per bench step, Philox noise in-kernel")


def run_reference(args, rank):
    if rank != 0:
        return
    # bounded sample of the same workload: same net, same SDE; ~10-30 s of CPU work per bench step
    n, s = 65536, 100
    for _ in range(min(args.warmup, 1)):
        cpu_sampler_rate(2048, 4)
    secs = []
    cores, kind = os.cpu_count(), "port"
    for _ in range(args.steps):
        _, cores, dt, kind = cpu_sampler_rate(n, s)
        secs.append(dt)
    value = n * s * len(secs) / sum(secs)
    what = ("the reference's own CDE.__call__ (baseline/_ref, unmodified models/diffusion.py + sdes.py + nets.py)"
            if kind == "reference" else "oracle port of models/diffusion.py:27-46 (baseline/_ref missing)")
    emit({
        "impl": "reference", "metric": "score-net evals/sec (posterior sampler)", "value": value, "unit": "evals/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(secs) / len(secs),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args) if args.workload in WORKLOADS else args.workload,
                   "sample": f"CPU step = {n} particles x {s} SDE steps of the synthetic CDE net (xdim 100, ydim 27) through "
                             f"{what}; the rate is linear in particles x steps (SURVEY.md App. B)"},
        "cpu_baseline": {"value": value, "unit": "evals/s", "cores": cores, "kind": kind,
                         "sample": f"{n} particles x {s} steps, torch CPU fp32, {cores} threads"},
        "e2e": {"value": value, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


# ----------------------------------------------------------------------------------------------- our arm
def setup_dist(world):
    import torch
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return local, dist


def require_lib():
    import dmip
    if not dmip.is_available():
        raise RuntimeError("libdmip_sm100.so missing or device is not sm_100 — no fallback")


def event_ms(fn, steps, warmup, before=None):
    """mean milliseconds per call of fn (CUDA events on torch's current stream = the stream the kernels launch on)"""
    import torch
    for _ in range(warmup):
        if before:
            before()
        fn()
    torch.cuda.synchronize()
    evs = []
    for _ in range(steps):
        if before:
            before()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        evs.append((e0, e1))
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in evs) / steps


def make_sampler_model(workload, rank=0):
    import torch
    from dmip.models import diffusion as dm
    kind, xdim, ydim, n_obs, n_def, s_def = WORKLOADS[workload]
    torch.manual_seed(0)
    cls = {"CDE": dm.CDE, "CDiffE": dm.CDiffE, "Posterior": dm.PosteriorDiffusionEstimator}[kind]
    model = cls(xdim, ydim, HIDDEN)          # default nn.Linear init under seed 0 (random-init weights, synthetic)
    model.sde.eval()
    y_host = torch.randn(n_obs, ydim, generator=torch.Generator().manual_seed(1 + rank))
    y_host = (y_host[0] if n_obs == 1 else y_host).contiguous().pin_memory()
    return model, y_host


def also_sampler(workload, N, S, flush, steps=1, warmup=1, e2e=True):
    """one short device-timed + one end-to-end run of a sampler workload (single GPU)"""
    import torch
    kind, xdim, ydim, n_obs, _, _ = WORKLOADS[workload]
    model, y_host = make_sampler_model(workload)
    y_dev = y_host.cuda()
    kw = dict(num_samples=N, num_steps=S, precision="bf16", seed=1234)
    ms = event_ms(lambda: model(y_dev, return_tensor=True, **kw), steps, warmup, before=flush.zero_)
    evals = float(n_obs) * N * S
    F = flop_per_eval(kind, xdim, ydim)
    out = {"config": f"{CFG_NAMES[workload]} xdim={xdim} ydim={ydim}, {n_obs} obs x {N} particles x {S} steps",
           "value": evals / (ms * 1e-3), "unit": "evals/s", "ms": ms, "samples_per_sec": evals / S / (ms * 1e-3),
           "dtype": "bf16" if model.last_precision == "bf16" else "f32", "gpu_launches": model.last_launch_count * steps,
           "roofline": tensor_roofline(evals * F / (ms * 1e-3) / 1e12, sustained=ms > 500, flop_per_eval=F,
                                       kernel="k_tc_mlp")}
    tr = load_traffic().get("k_tc_mlp_dram_bytes_per_launch", {})
    if workload in tr and N == WORKLOADS[workload][4] and S == WORKLOADS[workload][5]:
        out["roofline"]["traffic"] = tr[workload]
    if e2e:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        x_np = model(y_host, **kw)
        dt = time.perf_counter() - t0
        out["e2e"] = {"value": evals / dt, "unit": "evals/s", "h2d_bytes_per_step": n_obs * ydim * 4,
                      "d2h_bytes_per_step": int(x_np.size) * 4}
        del x_np
    del model
    torch.cuda.empty_cache()
    return out


def linear_batch(B, seed):
    import torch
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, 2, generator=g)
    A = torch.tensor([[1.0, 0.5], [0.0, 1.0]])
    y = x @ A.T + torch.tensor([0.3, 0.5]) + 0.3 * torch.randn(B, 2, generator=g)
    t = torch.rand(B, 1, generator=g) * 0.998 + 1e-3
    return x, y, t


def also_train(kind, B, steps=5, warmup=3, dist=None, rank=0, world=1):
    """configs[1]: linear CDE training step (fused loss forward + backward + Adam) at batch B per GPU.
    kind 'PINN': PINNLoss(FPE exact divergence, L1, ic L2) as config_linear.yml:11-16; 'DSM': the DSM branch."""
    import torch
    from dmip import distributed as dd, losses as dl
    from dmip.models.diffusion import CDE
    torch.manual_seed(0)
    model = CDE(2, 2, HIDDEN)
    opt = torch.optim.Adam(model.sde.a.parameters(), lr=1e-4, fused=True)   # config_linear.yml: Adam, lr 1e-4 (one fused launch)
    x, y, t = linear_batch(B, 7 + rank)
    xh, yh = x.pin_memory(), y.pin_memory()
    xd, yd, td = x.cuda(), y.cuda(), t.cuda()
    if kind == "PINN":
        loss_fn = dl.PINNLoss(lambda xx, yy: -xx, lam=0.001, lam2=0.1, pde_loss="FPE", ic_metric="L2", pde_metric="L1")
        flop_sample, name = 14, "configs[1]: linear CDE + PINNLoss(FPE exact divergence, L1, ic L2)"
    else:
        loss_fn = dl.DSMLoss()
        flop_sample, name = 3, "linear CDE + DSMLoss"
    F = flop_per_eval("CDE", 2, 2)
    last = {}

    def step(xa, ya):
        last["loss"], _ = dd.train_step_data_parallel(model, opt, loss_fn, xa, ya, td, batch_global=B * world)

    if dist is not None:
        dist.barrier()
    ms = event_ms(lambda: step(xd, yd), steps, warmup)
    launches = getattr(loss_fn, "last_launch_count", 0) * steps
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        step(xh.cuda(non_blocking=True), yh.cuda(non_blocking=True))
        lv = last["loss"].item()                        # device -> host read of the step's result
    e2e_s = time.perf_counter() - t0
    if dist is not None:
        tmax = torch.tensor([ms, e2e_s], device="cuda", dtype=torch.float64)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms, e2e_s = tmax.tolist()
    value = B * world / (ms * 1e-3)
    tc_path = os.environ.get("DMIP_LOSS_PATH", "tc") != "ffma"
    ach = value / world * flop_sample * F / 1e12
    if tc_path:
        roof = tensor_roofline(ach, sustained=False, flop_per_sample=flop_sample * F,
                               kernel="k_tcl_fwd + k_tcl_bwd + k_tcl_wgrad (bf16x3 split: 3 tensor-core FLOP per algorithmic FLOP)",
                               tensor_flops_issued_tflops=3 * ach)
        tr = load_traffic().get("k_tcl_dram_bytes_per_step", {})
        roof["traffic"] = tr.get(kind.lower()) if B == 65536 else None
    else:
        pk = measured_fp32_tflops()
        roof = {"bound": "tensor", "achieved": ach, "peak": pk, "unit": "TFLOP/s", "frac": ach / pk, "traffic": None,
                "peak_source": "measured cuBLAS SGEMM (TF32 off) on this GPU: the FFMA loss kernels are fp32",
                "flop_per_sample": flop_sample * F, "kernel": "k_jets_fwd + k_jets_bwd + k_wgrad"}
    out = {"config": f"{name}, batch {B} per GPU, Adam" + (f", data parallel over {world} GPUs (NCCL all-reduce of one "
                                                            f"gradient bucket)" if world > 1 else ""),
           "value": value, "unit": "samples/s", "ms": ms, "dtype": "bf16x3 (fp32-accurate split)" if tc_path else "f32",
           "loss": lv, "gpu_launches": launches, "roofline": roof,
           "e2e": {"value": B * world * steps / e2e_s, "unit": "samples/s", "h2d_bytes_per_step": B * 16,
                   "d2h_bytes_per_step": 4}}
    del model, opt
    torch.cuda.empty_cache()
    return out


def also_config0(batch=1000, n_batches=90, cpu_batches=12):
    """BASELINE configs[0]: the linear toy problem, CDiffE with the DSM loss, at the sizes of config/config_linear.yml
    (batch 1000, 90 000 training rows -> 90 batches per epoch, Adam lr 1e-4) through the drop-in `model.train_epoch`:
    at this batch a step is a handful of short launches, so what is measured is the host path (`graph=True`: the t draw,
    the noise draw and the fused loss kernels of a batch are ONE replay of a captured step, then the stock Adam step on
    the gradient bucket — no autograd round trip; 0.31 ms per step against 0.41 ms eager on the bench host).  The same epoch body of the stock
    reference classes runs on the host cores for `cpu_batches` batches."""
    import torch
    from dmip import losses as dl
    from dmip.models.diffusion import CDiffE
    torch.manual_seed(0)
    model = CDiffE(2, 2, HIDDEN)
    opt = torch.optim.Adam(model.sde.a.parameters(), lr=1e-4)      # the reference's optimizer (main_diffusion_linear.py:160)
    x, y, _ = linear_batch(batch * n_batches, 7)
    xd, yd = x.cuda(), y.cuda()

    def loader():
        for i in range(0, xd.shape[0], batch):
            yield xd[i:i + batch], yd[i:i + batch]

    loss_fn = dl.DSMLoss()
    for _ in range(2):                                             # warm-up epochs (Adam state, bucket, the captured step)
        model.train_epoch(opt, loss_fn, loader, graph=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    loss, _ = model.train_epoch(opt, loss_fn, loader, graph=True)
    lv = float(loss)                                               # device -> host read of the epoch's result
    dt = time.perf_counter() - t0
    out = {"config": f"configs[0]: linear CDiffE + DSMLoss, config_linear.yml sizes: one train_epoch of {n_batches} batches "
                     f"of {batch} (wall clock through model.train_epoch(..., graph=True): each batch one replay of the captured step + the "
                     f"stock Adam step; data resident on the GPU as in the reference's loader)",
           "value": batch * n_batches / dt, "unit": "samples/s", "ms": dt / n_batches * 1e3, "dtype": "bf16x3 (fp32-accurate split)",
           "loss": lv, "gpu_launches": getattr(loss_fn, "last_launch_count", 0) * n_batches,
           "roofline": {"bound": "host", "achieved": None, "peak": None, "unit": "ms/step", "frac": None, "traffic": None,
                        "note": "launch-bound: ~0.15 ms of kernels per step; see tools/small_batch_steps.py"},
           "e2e": {"value": batch * n_batches / dt, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    del model, opt
    ref = _reference_cde(2, 2, "CDiffE")
    if ref is not None:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        ropt = torch.optim.Adam(ref.sde.a.parameters(), lr=1e-4)
        rloss = ref.ref_losses.DSMLoss()

        def cpu_loader(nb):
            return lambda: ((x[i:i + batch], y[i:i + batch]) for i in range(0, nb * batch, batch))

        ref.train_epoch(ropt, rloss, cpu_loader(2))                # warm-up
        t0 = time.perf_counter()
        ref.train_epoch(ropt, rloss, cpu_loader(cpu_batches))
        cdt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": batch * cpu_batches / cdt, "unit": "samples/s", "cores": cores, "kind": "reference",
                               "ms_per_step": cdt / cpu_batches * 1e3,
                               "sample": f"{cpu_batches} batches of {batch}: the stock reference CDiffE.train_epoch + DSMLoss, torch CPU fp32"}
    return out


def also_posterior_loss(B=16384, steps=5, warmup=3):
    """PosteriorDiffusionEstimator.train_epoch body (models/diffusion.py:204-229): PosteriorLoss forward + backward +
    Adam on both nets, scatterometry shapes, random-init surrogate of the reference's architecture."""
    import torch
    from dmip.models.diffusion import PosteriorDiffusionEstimator
    torch.manual_seed(0)
    fm = torch.nn.Sequential(torch.nn.Linear(3, 256), torch.nn.ReLU(), torch.nn.Linear(256, 256), torch.nn.ReLU(),
                             torch.nn.Linear(256, 256), torch.nn.ReLU(), torch.nn.Linear(256, 23)).cuda()
    for q in fm.parameters():
        q.requires_grad = False
    m = PosteriorDiffusionEstimator(3, 23, HIDDEN)
    opt = torch.optim.Adam(m.sde.a.parameters(), lr=1e-4, fused=True)
    loss_fn = m.loss_fn(fm, 0.2, 0.01, lam=0.01)
    g = torch.Generator().manual_seed(3)
    x = (torch.rand(B, 3, generator=g) * 2 - 1)
    xh = x.pin_memory()
    xd = x.cuda()
    with torch.no_grad():
        yd = fm(xd)
    yh = yd.cpu().pin_memory()
    td = (torch.rand(B, 1, generator=g) * 0.998 + 1e-3).cuda()
    last = {}

    def step(xa, ya):
        loss, _ = loss_fn(m.sde, xa, ya, td)
        opt.zero_grad()
        loss.backward()
        opt.step()
        last["loss"] = loss.detach()

    ms = event_ms(lambda: step(xd, yd), steps, warmup)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        step(xh.cuda(non_blocking=True), yh.cuda(non_blocking=True))
        lv = last["loss"].item()
    e2e_s = time.perf_counter() - t0
    Fp, Fl = flop_per_eval("CDE", 0, 3) if False else 2 * (4 * 512 + 2 * 512 * 512 + 512 * 3), flop_per_eval("CDE", 3, 23)
    flop = 6 * Fp + 3 * Fl + SURR_FLOP       # prior: 1 + 3 tangent streams forward + 2 F backward; likelihood 3 F; surrogate VJP
    ach = B / (ms * 1e-3) * flop / 1e12
    return {"config": f"scatterometry DPS: PosteriorLoss forward + backward + Adam on prior and likelihood net, batch {B}",
            "value": B / (ms * 1e-3), "unit": "samples/s", "ms": ms, "dtype": "bf16x3 (fp32-accurate split)", "loss": lv,
            "gpu_launches": getattr(loss_fn, "last_launch_count", 0) * steps,
            "roofline": tensor_roofline(ach, sustained=False, flop_per_sample=flop,
                                        kernel="2 x (k_tcl_fwd + k_tcl_bwd + k_tcl_wgrad) + k_surrogate"),
            "e2e": {"value": B * steps / e2e_s, "unit": "samples/s", "h2d_bytes_per_step": B * (3 + 23) * 4,
                    "d2h_bytes_per_step": 4}}


def also_surrogate(rows=256 * 65536, steps=3, warmup=2):
    """K4 at the size of configs[3]: energy and posterior score (get_log_posterior + energy_grad) for 256 x 65,536 rows"""
    import torch
    from dmip import utils_scatterometry as us
    torch.manual_seed(0)
    fm = torch.nn.Sequential(torch.nn.Linear(3, 256), torch.nn.ReLU(), torch.nn.Linear(256, 256), torch.nn.ReLU(),
                             torch.nn.Linear(256, 256), torch.nn.ReLU(), torch.nn.Linear(256, 23)).cuda()
    for q in fm.parameters():
        q.requires_grad = False
    g = torch.Generator().manual_seed(5)
    chunk = 1 << 22                                   # the call is row-independent: 4M-row calls keep the host buffers small
    n_chunks = (rows + chunk - 1) // chunk
    xh = (torch.rand(chunk, 3, generator=g) * 2 - 1).pin_memory()
    xd = xh.cuda()
    with torch.no_grad():
        yd = fm(xd[:chunk // 65536]).contiguous()         # one observation per 65,536 rows (rows_per_obs of the C ABI)
    yh = yd.cpu().pin_memory()

    def call(xa, ya):
        return us.surrogate_call(fm, xa, ya, 0.2, 0.01, 1000.0)

    ms = event_ms(lambda: [call(xd, yd) for _ in range(n_chunks)], steps, warmup)
    gh = torch.empty(chunk, 3).pin_memory()           # the score comes back into pinned host memory
    eh = torch.empty(chunk).pin_memory()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n_chunks):
        E, gr, _ = call(xh.cuda(non_blocking=True), yh.cuda(non_blocking=True))
        gh.copy_(gr, non_blocking=True)
        eh.copy_(E, non_blocking=True)
        torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    ach = rows / (ms * 1e-3) * SURR_FLOP / 1e12
    ffma = os.environ.get("DMIP_SURROGATE_PATH") == "ffma"
    if ffma:
        pk = measured_fp32_tflops()
        roof = {"bound": "tensor", "achieved": ach, "peak": pk, "unit": "TFLOP/s", "frac": ach / pk, "traffic": None,
                "peak_source": "measured cuBLAS SGEMM (TF32 off) on this GPU (DMIP_SURROGATE_PATH=ffma: the fp32 FFMA kernel)",
                "flop_per_row": SURR_FLOP, "kernel": "k_surrogate"}
    else:
        # the two 256 x 256 layers (forward + reverse: 524,288 of the 550,912 FLOP / row) and the output layer run as
        # bf16x3 split products on the tensor cores: 3 issued FLOP per algorithmic FLOP
        roof = tensor_roofline(ach, sustained=False, flop_per_row=SURR_FLOP,
                               kernel="k_surrogate_tc (bf16x3 split: 3 tensor-core FLOP per algorithmic FLOP)",
                               tensor_flops_issued_tflops=3 * ach)
        tr = load_traffic().get("k_surrogate_tc_dram_bytes_per_launch", {})
        roof["traffic"] = tr.get(f"{chunk}_rows")          # per launch (one 4M-row call), like `achieved`'s launch duration
    return {"config": f"K4 surrogate energy + score, {rows} rows (256 observations x 65,536 particles), in calls of {chunk} rows",
            "value": rows / (ms * 1e-3), "unit": "rows/s", "ms": ms, "dtype": "f32" if ffma else "bf16x3",
            "gpu_launches": n_chunks * steps * (5 if ffma else 2), "roofline": roof,
            "e2e": {"value": rows / e2e_s, "unit": "rows/s", "h2d_bytes_per_step": rows * 3 * 4 + (rows // 65536) * 23 * 4, "d2h_bytes_per_step": rows * 16}}


def run_also(args, flush):
    """The other BASELINE configs, single GPU, short runs; every entry carries value / ms / roofline / e2e."""
    import torch
    also = {}

    def guard(name, fn):
        try:
            also[name] = fn()
        except Exception as e:                         # noqa: BLE001 — one failing extra must not lose the headline
            also[name] = {"error": repr(e)[:300]}
        torch.cuda.empty_cache()

    guard("config0_linear_cdiffe_dsm", also_config0)
    guard("cdiffe_scat", lambda: also_sampler("cdiffe_scat", 1 << 20, 1000, flush))
    guard("dps_scat", lambda: also_sampler("dps_scat", 1 << 16, 1000, flush))
    guard("pinn_linear", lambda: also_train("PINN", 65536))
    guard("dsm_linear", lambda: also_train("DSM", 65536))
    guard("posterior_loss", also_posterior_loss)
    guard("surrogate_score", also_surrogate)
    sweep = {}
    for n in (1 << 16, 1 << 18, 1 << 22, 1 << 24):
        try:
            r = also_sampler("synthetic", n, 200, flush, steps=1, warmup=1, e2e=n <= (1 << 22))
            sweep[str(n)] = {"value": r["value"], "ms": r["ms"], "frac": r["roofline"]["frac"],
                             "e2e": r.get("e2e", {}).get("value")}
        except Exception as e:                         # noqa: BLE001
            sweep[str(n)] = {"error": repr(e)[:200]}
    also["sweep"] = {"config": "configs[4] synthetic CDE, particles swept at S = 200 SDE steps, 1 GPU (e2e up to 4M particles: "
                               "the 16M result is 6.7 GB of samples)", "unit": "evals/s", "particles": sweep}
    return also


def dump_rows(dirname, name, rows):
    """DIR/<name>.npy of a (n, d) CUDA tensor as float32; above DUMP_ROWS rows a fixed seeded sample of them, in row order"""
    import numpy as np
    import torch
    if rows.shape[0] > DUMP_ROWS:
        idx = np.sort(np.random.default_rng(0).choice(rows.shape[0], DUMP_ROWS, replace=False))
        rows = rows[torch.from_numpy(idx).to(rows.device)]
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, name + ".npy"), rows.float().cpu().numpy())


def run_sampler(args, rank, world):
    import torch
    local, dist = setup_dist(world)
    require_lib()
    kind, xdim, ydim, n_obs, n_def, s_def = WORKLOADS[args.workload]
    N, S = args.particles or n_def, args.sde_steps or s_def
    F = flop_per_eval(kind, xdim, ydim)
    model, y_host = make_sampler_model(args.workload, rank)
    y_dev = y_host.cuda()
    per_rank = n_obs * N                      # particles integrated by one rank per bench step
    kw = dict(num_samples=N, num_steps=S, precision=args.precision, seed=1234, gidx_base=rank * per_rank)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 0)):
        flush.zero_()            # also warms the fill kernel: its first launch loads a torch module (up to 0.6 s, host side)
        model(y_dev, return_tensor=True, **kw)
    barrier()

    # ---- device-resident timing (CUDA events on the stream the kernel is launched on = torch's current stream)
    clocks = ClockSampler(local)
    time.sleep(0.25)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches = 0
    t_wall0 = time.time()
    barrier()
    ev0.record()
    for i in range(args.steps):
        flush.zero_()                                                     # evict L2 between timed iterations
        kev[i][0].record()
        out = model(y_dev, return_tensor=True, **kw)
        kev[i][1].record()
        launches += model.last_launch_count
    ev1.record()
    barrier()
    t_wall1 = time.time()
    ms = ev0.elapsed_time(ev1)
    kernel_ms = sum(a.elapsed_time(b) for a, b in kev) / args.steps      # k_tc_mlp (+ the weight re-pack check): per launch
    gaps_ms = [ev0.elapsed_time(kev[0][0])] + [kev[i][1].elapsed_time(kev[i + 1][0]) for i in range(args.steps - 1)] + \
        [kev[-1][1].elapsed_time(ev1)]
    clk = clocks.stop(t_wall0, t_wall1)
    finite = bool(torch.isfinite(out).all().item())
    if args.dump_outputs and rank == 0:
        dump_rows(args.dump_outputs, "samples", out.reshape(-1, xdim))
    del out

    # ---- end-to-end through the reference-facing call, host buffers
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        x_np = model(y_host, **kw)                                        # H2D of y, D2H of the samples (numpy)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    assert x_np.shape[-1] == xdim
    del x_np

    if dist is not None:
        tmax = torch.tensor([ms, e2e_s, kernel_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms, e2e_s, kernel_ms = tmax.tolist()

    # ---- the other BASELINE configs (single GPU), or the data-parallel training step (multi GPU)
    also = None
    if not args.no_also and args.workload == "synthetic" and not args.particles and not args.sde_steps:
        if world == 1:
            also = run_also(args, flush)
        else:
            try:
                also = {"pinn_dp": also_train("PINN", 65536, dist=dist, rank=rank, world=world)}
            except Exception as e:                     # noqa: BLE001
                also = {"pinn_dp": {"error": repr(e)[:300]}}
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    evals = float(per_rank) * S * args.steps * world
    value = evals / (ms * 1e-3)
    ach_tf = (float(per_rank) * S / (kernel_ms * 1e-3)) * F / 1e12      # per GPU, from the kernel's own launch duration
    roof = tensor_roofline(ach_tf, sustained=True, flop_per_eval=F, kernel="k_tc_mlp (one launch per bench step)",
                           kernel_ms=kernel_ms)
    roof["peak_source"] += ": the kernel runs inside a > 1 s step"
    peaks = load_peaks()
    roof["frac_of_burst_peak"] = (ach_tf / peaks["bf16_tflops"]) if peaks.get("bf16_tflops") else None
    # measured for the default launch of a workload only (ncu capture of that exact command); null otherwise
    tr = load_traffic().get("k_tc_mlp_dram_bytes_per_launch", {})
    roof["traffic"] = tr.get(args.workload) if (not args.particles and not args.sde_steps) else None
    ran = getattr(model, "last_precision", args.precision)
    line = {
        "metric": "score-net evals/sec (posterior sampler)", "value": value, "unit": "evals/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if ran == "bf16" else "f32",     # the path that RAN: a bf16 request outside the tcgen05 kernel's shapes runs fp32
        "data": "synthetic",
        "config": {"workload": workload_name(args),
                   "samples_per_sec": value / S, "l2": "256 MB buffer zeroed between timed iterations",
                   "finite": finite, "gaps_ms": [round(g, 2) for g in gaps_ms]},
        "roofline": roof,
        "e2e": {"value": evals / e2e_s, "unit": "evals/s", "h2d_bytes_per_step": n_obs * ydim * 4,
                "d2h_bytes_per_step": per_rank * xdim * 4},
        "gpu_launches": launches,
        "clocks": clk,
    }
    if also is not None:
        line["also"] = also
    if not args.no_cpu_baseline and world == 1:
        n, s = 65536, 100
        r, cores, dt, kind = cpu_sampler_rate(n, s)
        line["cpu_baseline"] = {"value": r, "unit": "evals/s", "cores": cores, "kind": kind,
                                "sample": f"{n} particles x {s} steps of the synthetic CDE net, torch CPU fp32, {dt:.1f} s"
                                          + (" (stock reference CDE.__call__)" if kind == "reference" else " (oracle port)")}
    emit(line)
    if dist is not None:
        dist.destroy_process_group()


def run_single(args, rank, world, fn, metric, **kw):
    """a non-sampler workload as the JSON line's headline"""
    local, dist = setup_dist(world)
    require_lib()
    r = fn(dist=dist, rank=rank, world=world, **kw) if fn is also_train else fn(**kw)
    if dist is not None:
        dist.destroy_process_group()
    if rank != 0:
        return
    emit({"metric": metric, "value": r["value"], "unit": r["unit"], "n_gpus": world, "steps": args.steps,
          "warmup": args.warmup, "ms_per_step": r["ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
          "dtype": r["dtype"], "data": "synthetic", "config": {"workload": r["config"], "loss": r.get("loss")},
          "roofline": r["roofline"], "e2e": r["e2e"], "gpu_launches": r["gpu_launches"]})


def run_mcmc(args, rank, world):
    """Ground-truth generation for the scatterometry KL (generate_scatterometry_ground_truth.py): random-walk Metropolis
    chains on the surrogate posterior, 8 observations x 30,000 chains per GPU (config_scatterometry.yml: n_samples_x),
    METR_STEPS = 1000 per bench step, one kernel launch.  Observations shard over ranks, no collective."""
    import torch
    from dmip import mcmc
    local, dist = setup_dist(world)
    require_lib()
    torch.manual_seed(0)
    fm = torch.nn.Sequential(torch.nn.Linear(3, 256), torch.nn.ReLU(), torch.nn.Linear(256, 256), torch.nn.ReLU(),
                             torch.nn.Linear(256, 256), torch.nn.ReLU(), torch.nn.Linear(256, 23)).cuda()
    for q in fm.parameters():
        q.requires_grad = False
    n_obs, n_per, S = 8, args.particles or 30000, args.sde_steps or 1000
    g = torch.Generator().manual_seed(13 + rank)
    xt = (torch.rand(n_obs, 3, generator=g) * 2 - 1).cuda()
    with torch.no_grad():
        ys = fm(xt)
    ys_h = ys.cpu().pin_memory()
    x0 = (torch.rand(n_obs * n_per, 3, generator=g) * 2 - 1).cuda()

    def step(yv, to_host=False):
        x, _ = mcmc.anneal_to_energy(x0, fm, 0.2, 0.01, yv, 1000.0, S, 0.5, seed=1, gidx_base=rank * n_obs * n_per)
        return x.cpu() if to_host else x

    if dist is not None:
        dist.barrier()
    ms = event_ms(lambda: step(ys), args.steps, max(args.warmup, 0)) * args.steps
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step(ys_h.cuda(non_blocking=True), to_host=True)
    e2e_s = time.perf_counter() - t0
    if dist is not None:
        tmax = torch.tensor([ms, e2e_s], device="cuda", dtype=torch.float64)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms, e2e_s = tmax.tolist()
    pk = measured_fp32_tflops()
    if dist is not None:
        dist.destroy_process_group()
    if rank != 0:
        return
    F = 2 * (3 * 256 + 256 * 256 * 2 + 256 * 23)
    work = n_obs * n_per * S * world * args.steps
    value = work / (ms * 1e-3)
    ach = value / world * F / 1e12
    emit({
        "metric": "Metropolis chain-steps/sec (scatterometry ground truth)", "value": value, "unit": "chain-steps/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"scatterometry Metropolis ground truth: {n_obs} observations x {n_per} chains per GPU x {S} "
                               "steps per bench step, random-init surrogate 3-256-256-256-23, Philox in-kernel"},
        "roofline": {"bound": "tensor", "achieved": ach, "peak": pk, "unit": "TFLOP/s", "frac": ach / pk, "traffic": None,
                     "peak_source": "measured cuBLAS SGEMM (TF32 off) on this GPU: k_metropolis is fp32 FFMA",
                     "flop_per_chain_step": F, "kernel": "k_metropolis (one launch per bench step)"},
        "e2e": {"value": work / e2e_s, "unit": "chain-steps/s", "h2d_bytes_per_step": n_obs * 23 * 4,
                "d2h_bytes_per_step": n_obs * n_per * 12},
        "gpu_launches": getattr(mcmc.anneal_to_energy, "last_launch_count", 0) * args.steps,
    })


def main():
    args = parse()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if world > 1 and os.environ.get("NCCL_DEBUG", "VERSION").upper() in ("VERSION", "WARN"):
        os.environ["NCCL_DEBUG"] = "INFO"                # before torch / NCCL load: the communicator log (ranks, rings, NVLS)
                                                         # goes to stderr (claim_stdout), never into the JSON line
    claim_stdout()
    if args.impl == "reference":
        run_reference(args, rank)
    elif args.workload == "mcmc_scat":
        run_mcmc(args, rank, world)
    elif args.workload == "pinn_linear":
        run_single(args, rank, world, also_train, "PINNLoss training samples/sec", kind="PINN", B=args.particles or 65536,
                   steps=args.steps, warmup=args.warmup)
    elif args.workload == "dsm_linear":
        run_single(args, rank, world, also_train, "DSMLoss training samples/sec", kind="DSM", B=args.particles or 65536,
                   steps=args.steps, warmup=args.warmup)
    elif args.workload == "posterior_loss":
        run_single(args, rank, world, also_posterior_loss, "PosteriorLoss training samples/sec", B=args.particles or 16384,
                   steps=args.steps, warmup=args.warmup)
    elif args.workload == "surrogate_score":
        run_single(args, rank, world, also_surrogate, "surrogate score rows/sec", rows=args.particles or 256 * 65536,
                   steps=args.steps, warmup=args.warmup)
    else:
        run_sampler(args, rank, world)


if __name__ == "__main__":
    main()
