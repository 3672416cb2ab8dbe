"""Step time of the fused score-training losses under the VE-SDE against the VP-SDE, and of this build against an earlier
build of the library for the VP-SDE; and whether the VP losses and gradients of the two builds are bit-identical.

    python tools/ve_loss_bench.py --parent-lib PATH/libdmip_sm100.so [--reps 3] [--iters 20] [--out DIR]

Problems: linear CDE (xdim = ydim = 2, [512]^3 net), batch 65,536; DSM and PINN (Score-FPE, exact divergence, d = 2, the
forward-only route; ic L2, pde L1), on the tcgen05 kernels (the default dispatch) and the FFMA kernels
(DMIP_LOSS_PATH=ffma).  One fused call = the forward and backward kernels of the loss and the parameter gradient.  Each
build runs in a process of its own (the library is chosen by DMIP_LIB); the builds alternate, `reps` rounds, and each
round times `iters` calls with CUDA events after 3 warm-up calls.  Reported: the median over rounds of the per-call time,
the spread (min, max) of the round times, the GPU name and power limit read in the same run.  The earlier build only runs
VP (it has no VE-SDE).

Outputs: the loss and every parameter gradient of the last warm-up call of each round.  The kernels reduce the loss and
the split-K weight gradients with fp32 atomics, whose order varies from run to run, so each comparison of the two builds
is reported beside the same comparison of one build with itself (round 0 against the later rounds): bitwise equal, or the
largest difference relative to each tensor's largest entry.  At batch 1 (one tile, one split: no reordering) the same
outputs are also kept, and there the two builds must agree bit for bit."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROBLEMS = [(loss, path) for loss in ("DSM", "PINN") for path in ("tc", "ffma")]


def worker(sdes_to_run, iters, dump):
    sys.path.insert(0, ROOT)
    import torch
    from dmip import losses as dl, sdes
    from dmip.linear_problem import LinearForwardProblem
    from dmip.models.diffusion import CDE
    dev = "cuda"
    B = 65536
    lin = LinearForwardProblem()
    g = torch.Generator().manual_seed(7)
    x = torch.randn(B, 2, generator=g)
    y = lin(x) + 0.3 * torch.randn(B, 2, generator=g)
    t = torch.rand(B, 1, generator=g) * (1 - 2e-4) + 1e-4
    eps = torch.randn(B, 2, generator=g)
    ic = lin.score_posterior(x, y).to(dev)
    x, y, t, eps = (v.to(dev) for v in (x, y, t, eps))
    res, outs = {}, {}
    for sde_name in sdes_to_run:
        torch.manual_seed(0)
        base = sdes.VarianceExplodingSDE(sigma_min=0.05, sigma_max=4.0) if sde_name == "VE" else None
        m = CDE(2, 2, [512, 512, 512], base_sde=base)
        m.sde.to(dev)
        for loss_name, path in PROBLEMS:
            os.environ["DMIP_LOSS_PATH"] = path
            if loss_name == "DSM":
                def call():
                    return dl.dsm_fused(m, x, y, t, eps)[0]
            else:
                fn = dl.PINNLoss(lambda xx, yy: ic, lam=0.001, lam2=0.1, pde_loss="FPE", ic_metric="L2", pde_metric="L1")

                def call():
                    return fn(m.sde, x, y, x, t, eps, None, None)[0]
            for _ in range(3):
                m.sde.a.zero_grad(set_to_none=True)
                loss = call()
                loss.backward()
            outs[f"{sde_name}/{loss_name}/{path}"] = ([loss.detach().cpu()] +
                                                      [p.grad.detach().cpu().clone() for p in m.sde.a.parameters()])
            one = [v[:1] for v in (x, y, t, eps)]
            m.sde.a.zero_grad(set_to_none=True)
            if loss_name == "DSM":
                l1 = dl.dsm_fused(m, *one)[0]
            else:
                fn1 = dl.PINNLoss(lambda xx, yy: ic[:1], lam=0.001, lam2=0.1, pde_loss="FPE", ic_metric="L2",
                                  pde_metric="L1")
                l1 = fn1(m.sde, one[0], one[1], one[0], one[2], one[3], None, None)[0]
            l1.backward()
            outs[f"{sde_name}/{loss_name}/{path}/B1"] = ([l1.detach().cpu()] +
                                                         [p.grad.detach().cpu().clone() for p in m.sde.a.parameters()])
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                loss = call()
            e1.record()
            torch.cuda.synchronize()
            res[f"{sde_name}/{loss_name}/{path}"] = e0.elapsed_time(e1) / iters
            os.environ.pop("DMIP_LOSS_PATH", None)
    torch.save(outs, dump)
    return res


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None, help="directory for the log (default: print only)")
    ap.add_argument("--worker", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--sdes", default="VP,VE", help=argparse.SUPPRESS)
    ap.add_argument("--dump", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker:
        print(json.dumps(worker(a.sdes.split(","), a.iters, a.dump)))
        return
    import torch
    builds = {"new": os.path.join(ROOT, "diffusion-modelling-for-inverse-problems_b200", "libdmip_sm100.so"),
              "parent": os.path.abspath(a.parent_lib)}
    times = {}
    lines = [f"gpu: {gpu_info()}", f"batch 65536, linear CDE 2+2, [512]^3; {a.iters} calls per round, {a.reps} rounds, "
             "builds alternated; ms per fused loss call (forward + backward + parameter gradient)"]
    with tempfile.TemporaryDirectory() as td:
        dumps = {"new": [], "parent": []}
        for r in range(a.reps):
            for name in (("new", "parent") if r % 2 == 0 else ("parent", "new")):
                dump = os.path.join(td, f"{name}.pt")
                env = dict(os.environ, DMIP_LIB=builds[name])
                cmd = [sys.executable, os.path.abspath(__file__), "--parent-lib", a.parent_lib, "--worker", name,
                       "--iters", str(a.iters), "--sdes", "VP,VE" if name == "new" else "VP", "--dump", dump]
                out = subprocess.run(cmd, env=env, capture_output=True, text=True, cwd=ROOT)
                if out.returncode:
                    raise SystemExit(f"worker {name} failed:\n{out.stdout}\n{out.stderr}")
                for k, v in json.loads(out.stdout.strip().splitlines()[-1]).items():
                    times.setdefault(f"{name}:{k}", []).append(v)
                dumps[name].append(torch.load(dump))

        def diff(u, v):
            """(bitwise equal, largest |u - v| relative to each tensor's largest |v|)"""
            same = len(u) == len(v) and all(torch.equal(p, q) for p, q in zip(u, v))
            rel = max(((p.double() - q.double()).abs().max() / q.double().abs().max().clamp_min(1e-30)).item()
                      for p, q in zip(u, v))
            return same, rel
        cmp = {}
        for k in dumps["parent"][0]:
            across = [diff(dumps["new"][r][k], dumps["parent"][r][k]) for r in range(a.reps)]
            par = [diff(dumps["parent"][r][k], dumps["parent"][0][k]) for r in range(1, a.reps)]
            own = [diff(dumps["new"][r][k], dumps["new"][0][k]) for r in range(1, a.reps)]
            cmp[k] = (across, par, own)
        for k, v in dumps["new"][0].items():
            lines.append(f"finite {k}: {all(bool(torch.isfinite(u).all()) for u in v)}  loss {v[0].item():.6g}")
    for k in sorted(times):
        v = times[k]
        lines.append(f"{k:28s} median {statistics.median(v):8.4f} ms   rounds min {min(v):8.4f}  max {max(v):8.4f}")
    fmt = lambda xs: ", ".join(f"{'equal' if s else f'{r:.1e}'}" for s, r in xs) or "-"
    for k, (across, par, own) in sorted(cmp.items()):
        lines.append(f"{k}: new vs parent per round [{fmt(across)}]; parent vs its round 0 [{fmt(par)}]; "
                     f"new vs its round 0 [{fmt(own)}]")
    text = "\n".join(lines)
    print(text)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "ve_loss_bench.log"), "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
