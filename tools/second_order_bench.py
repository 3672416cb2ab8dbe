"""Step time of the reference's literal Score-FPE PINN loss (autograd double backward through the score net) on the
library's nets, on the plain torch module chain and as the fused PINNLoss; and the fused DSM / PINN steps of this build
against an earlier build of the library.

    python tools/second_order_bench.py --parent-lib PATH/libdmip_sm100.so [--reps 3] [--out DIR]

Workload: linear CDE (xdim = ydim = 2, [512]^3 net), batch 1,000 and 65,536, one training step = the loss and
`loss.backward()` (parameter gradients), ic L2, pde L2, exact divergence.  Arms:
  (a) literal  — the loss as losses.py:77-98 / :214-242 write it (d create_graph calls for div s, grad_x from a second-order
                 call, ds/dt through a t leaf) through dmip.nets.MLP: forward with stash, backward and double backward on
                 the tcgen05 loss kernels;
  (b) chain    — the same loss through the plain torch module chain on the same weights (fp32, TF32 off);
  (c) fused    — dmip.losses.PINNLoss (forward-mode jets, one fused call), for scale.
The arms alternate inside each round; `reps` rounds; each round times `iters` steps with CUDA events after 2 warm-up steps.
The A/B part runs the fused DSM and PINN steps at 65,536 in one process per build, builds alternated (DMIP_LIB chooses the
library).  Reported: medians over rounds and the (min, max) of the round times, GPU name and power limit of the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _problem(B, dev):
    import torch
    from dmip.linear_problem import LinearForwardProblem
    lin = LinearForwardProblem()
    g = torch.Generator().manual_seed(7)
    x = torch.randn(B, 2, generator=g)
    y = lin(x) + 0.3 * torch.randn(B, 2, generator=g)
    t = torch.rand(B, 1, generator=g) * (1 - 2e-4) + 1e-4
    eps = torch.randn(B, 2, generator=g)
    ic = lin.score_posterior(x, y)
    return [v.to(dev) for v in (x, y, t, eps, ic)]


def literal_pinn(apply, x, y, t, eps, ic, lam=0.001, lam2=0.1):
    """PINNLoss with the Score-FPE residual built by autograd (CDE: z = x, cond = y), `apply(z, cond, t)` = the net"""
    import torch
    from oracle import losses as ol, vp
    t = t.detach().clone().requires_grad_(True)
    std = vp.var(t) ** 0.5
    z_t = vp.mean_weight(t) * x + std * eps
    beta = vp.beta(t)
    s = apply(z_t, y, t) / beta ** 0.5
    n, d = s.shape
    div = sum(torch.autograd.grad(s[:, k].sum(), z_t, create_graph=True)[0][:, k] for k in range(d)).reshape(n, 1)
    phi = div + (s ** 2).sum(1, keepdim=True) + (z_t * s).sum(1, keepdim=True)
    grad_x = torch.autograd.grad(phi.sum(), z_t, retain_graph=True)[0].detach()
    ds_dt = torch.cat([torch.autograd.grad(s[:, i].sum(), t, create_graph=True)[0] for i in range(d)], 1)
    t0 = torch.zeros_like(t)
    s0 = apply(x, y, t0) / vp.beta(t0) ** 0.5
    terms = {"s": s, "beta": beta, "ds_dt": ds_dt, "div_s": div, "grad_x": grad_x}
    l_ic = lam2 * ((s0 - ic) ** 2).mean(1, keepdim=True)
    l_pde = lam * ol.score_fpe(terms, "L2")
    return ol.dsm(s, std, eps).mean() + l_ic.mean() + l_pde.mean()


def _time(step, iters):
    import torch
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        step()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def worker_arms(reps):
    sys.path.insert(0, ROOT)
    import torch
    from dmip import losses as dl
    from dmip.models.diffusion import CDE
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    dev = "cuda"
    torch.manual_seed(0)
    m = CDE(2, 2, [512, 512, 512])
    m.sde.to(dev)
    net = m.sde.a

    def chain(z, cond, t):
        return torch.nn.Sequential.forward(net, torch.cat([z, cond, t.reshape(-1, 1)], 1))

    res, losses = {}, {}
    for B in (1000, 65536):
        x, y, t, eps, ic = _problem(B, dev)
        fused = dl.PINNLoss(lambda xx, yy: ic, lam=0.001, lam2=0.1, pde_loss="FPE", ic_metric="L2", pde_metric="L2")
        arms = {"literal": lambda: literal_pinn(net, x, y, t, eps, ic),
                "chain": lambda: literal_pinn(chain, x, y, t, eps, ic),
                "fused": lambda: fused(m.sde, x, y, x, t, eps, None, None)[0]}
        iters = 20 if B <= 1000 else 5
        for r in range(reps):
            for name in (list(arms) if r % 2 == 0 else list(arms)[::-1]):
                def step(f=arms[name]):
                    net.zero_grad(set_to_none=True)
                    loss = f()
                    loss.backward()
                res.setdefault(f"B{B}/{name}", []).append(_time(step, iters))
        for name, f in arms.items():
            net.zero_grad(set_to_none=True)
            loss = f()
            loss.backward()
            losses[f"B{B}/{name}"] = [loss.item(), sum(float(p.grad.double().norm() ** 2) for p in net.parameters()) ** 0.5]
    return {"times": res, "values": losses}


def worker_fused():
    sys.path.insert(0, ROOT)
    import torch
    from dmip import losses as dl
    from dmip.models.diffusion import CDE
    dev = "cuda"
    torch.manual_seed(0)
    m = CDE(2, 2, [512, 512, 512])
    m.sde.to(dev)
    x, y, t, eps, ic = _problem(65536, dev)
    fn = dl.PINNLoss(lambda xx, yy: ic, lam=0.001, lam2=0.1, pde_loss="FPE", ic_metric="L2", pde_metric="L1")
    steps = {"DSM": lambda: dl.dsm_fused(m, x, y, t, eps)[0], "PINN": lambda: fn(m.sde, x, y, x, t, eps, None, None)[0]}
    res = {}
    for name, f in steps.items():
        def step(f=f):
            m.sde.a.zero_grad(set_to_none=True)
            f().backward()
        res[name] = _time(step, 20)
    return res


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="directory for the log (default: print only)")
    ap.add_argument("--worker", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker == "arms":
        print(json.dumps(worker_arms(a.reps)))
        return
    if a.worker == "fused":
        print(json.dumps(worker_fused()))
        return
    builds = {"new": os.path.join(ROOT, "diffusion-modelling-for-inverse-problems_b200", "libdmip_sm100.so"),
              "parent": os.path.abspath(a.parent_lib)}

    def run(worker, build):
        cmd = [sys.executable, os.path.abspath(__file__), "--parent-lib", a.parent_lib, "--worker", worker,
               "--reps", str(a.reps)]
        out = subprocess.run(cmd, env=dict(os.environ, DMIP_LIB=builds[build]), capture_output=True, text=True, cwd=ROOT)
        if out.returncode:
            raise SystemExit(f"worker {worker} ({build}) failed:\n{out.stdout}\n{out.stderr}")
        return json.loads(out.stdout.strip().splitlines()[-1])

    lines = [f"gpu: {gpu_info()}",
             "literal Score-FPE PINN step (loss + backward), linear CDE 2+2, [512]^3, exact divergence; ms per step, "
             f"median of {a.reps} alternated rounds (min, max)"]
    arms = run("arms", "new")
    for k in sorted(arms["times"]):
        v = arms["times"][k]
        lines.append(f"{k:16s} median {statistics.median(v):9.3f} ms   rounds min {min(v):9.3f}  max {max(v):9.3f}")
    for k in sorted(arms["values"]):
        lines.append(f"{k:16s} loss {arms['values'][k][0]:.6g}  |grad| {arms['values'][k][1]:.6g}")
    ab = {}
    for r in range(a.reps):
        for build in (("new", "parent") if r % 2 == 0 else ("parent", "new")):
            for k, v in run("fused", build).items():
                ab.setdefault(f"{build}:{k}", []).append(v)
    lines.append(f"fused steps at 65,536 (loss + backward), 20 steps per round, {a.reps} rounds, builds alternated")
    for k in sorted(ab):
        v = ab[k]
        lines.append(f"{k:16s} median {statistics.median(v):9.4f} ms   rounds min {min(v):9.4f}  max {max(v):9.4f}")
    text = "\n".join(lines)
    print(text)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "second_order_bench.log"), "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
