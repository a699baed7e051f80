"""K7-NB against K7: the fused negative-binomial call (gpz_negbin_fwdbwd_f32) and the dense Poisson call on the same inputs.

    python tools/bench_negbin.py OUTDIR [--reps 200] [--warmup 20]

Workloads, at config 2's shape (G = 2000, B = 32768, F = 10, E = 1, fp32):
  * the likelihood call alone, counts as fp32 and as uint8: milliseconds per call (CUDA events over --reps launches after --warmup,
    NB and Poisson alternated in three rounds, median of the rounds).  The inputs are replicated until the copies exceed 256 MB and
    the launches cycle through them, so no call reads y from the 126 MB L2;
  * one full config-2 model.elbo fwd+bwd step of NSF2_NB against NSF2 (same parameters, same counts), alternated the same way
    (--step-reps steps per round).
Every round's time is recorded next to the median, so the spread can be read off.
The GPU's name and power limit are read with nvidia-smi in the same run.  Writes OUTDIR/bench_negbin.json.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

L2_DEFEAT_BYTES = 256 << 20


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = [s.strip() for s in out.stdout.strip().splitlines()[0].split(",")]
    return dict(gpu=name, power_limit=power)


def _time(fns, reps, warmup, rounds=3):
    """Per-call milliseconds of each fn (called with the launch index) in each round, the fns alternated per round."""
    import torch
    res = {k: [] for k in fns}
    for k, fn in fns.items():
        for i in range(warmup):
            fn(i)
    torch.cuda.synchronize()
    for _ in range(rounds):
        for k, fn in fns.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(reps):
                fn(i)
            e1.record()
            torch.cuda.synchronize()
            res[k].append(e0.elapsed_time(e1) / reps)
    return res


def call_point(ydt, reps, warmup, G=2000, B=32768, F=10, E=1, seed=0):
    import torch
    from gpzoo_b200 import functional as Fn
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(seed)
    y = torch.poisson(2 * torch.rand(G, B, generator=g, device=dev)).to(ydt)
    copies = max(1, math.ceil(L2_DEFEAT_BYTES / (y.numel() * y.element_size())))
    ys = [y] + [y.clone() for _ in range(copies - 1)]
    W = torch.rand(G, F, generator=g, device=dev) - 1.0
    V = 1 + 0.2 * torch.randn(B, generator=g, device=dev)
    D = torch.randn(G, generator=g, device=dev)
    mean = 0.3 * torch.randn(F, B, generator=g, device=dev)
    var = 0.05 + 0.3 * torch.rand(F, B, generator=g, device=dev)
    eps = torch.randn(E, F, B, generator=g, device=dev)
    nb = lambda i: Fn.NegBinLL.apply(ys[i % copies], None, W, V, D, mean, var, eps, F, 5e-2, True, True)
    po = lambda i: Fn.PoissonLL.apply(ys[i % copies], None, W, V, mean, var, eps, F, 5e-2, True, True)
    with torch.no_grad():
        t = _time(dict(negbin=nb, poisson=po), reps, warmup)
    nb, po = statistics.median(t["negbin"]), statistics.median(t["poisson"])
    return dict(counts=str(ydt).replace("torch.", ""), y_copies=copies, negbin_ms=nb, poisson_ms=po, ratio=nb / po,
                negbin_rounds_ms=t["negbin"], poisson_rounds_ms=t["poisson"])


def step_point(reps, warmup):
    """config 2 (bench.py's problem): one NSF2_NB and one NSF2 elbo fwd+bwd, same parameters and counts."""
    import torch
    import gpzoo_b200 as gz
    from gpzoo_b200 import synthetic
    prob = synthetic.nsf_problem(N=32768, M=1024, L=10, G=2000, E=1, seed=0, coord_scale=100.0, lengthscale=1.7, jitter=0.1,
                                 dtype=torch.float32, device="cuda")
    models = {}
    for name, cls in (("negbin", gz.likelihoods.NSF2_NB), ("poisson", gz.likelihoods.NSF2)):
        kern = gz.kernels.NSF_RBF(L=10)
        kern.sigma, kern.lengthscale = torch.nn.Parameter(prob["sigma"].clone()), torch.nn.Parameter(prob["lengthscale"].clone())
        gp = gz.gp.SVGP(kern, dim=2, M=1024, jitter=prob["jitter"])
        gp.Z, gp.mu, gp.Lu = (torch.nn.Parameter(prob[k].clone()) for k in ("Z", "mu", "Lu_raw"))
        m = cls(gp, prob["y"], L=10).cuda()
        m.W, m.V = torch.nn.Parameter(prob["W"].clone()), torch.nn.Parameter(prob["V"].clone())
        models[name] = m
    X, y = prob["X"], prob["y"].to(torch.uint8)
    eps = torch.randn(1, 10, 32768, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))

    def step(m):
        def f(i):
            m.zero_grad(set_to_none=True)
            m.elbo(X, y, E=1, eps=eps).backward()
        return f
    gz.functional.set_sync_checks(False)
    t = _time({k: step(m) for k, m in models.items()}, reps, warmup)
    nb, po = statistics.median(t["negbin"]), statistics.median(t["poisson"])
    return dict(negbin_step_ms=nb, poisson_step_ms=po, ratio=nb / po, negbin_rounds_ms=t["negbin"], poisson_rounds_ms=t["poisson"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--step-reps", type=int, default=200)      # 200 steps of ~8 ms: a window of 1.6 s per round
    a = ap.parse_args()
    import torch
    res = dict(gpu_info(), shape=dict(G=2000, B=32768, F=10, E=1, dtype="float32"))
    res["calls"] = [call_point(torch.float32, a.reps, a.warmup), call_point(torch.uint8, a.reps, a.warmup)]
    res["step"] = step_point(a.step_reps, 5)
    os.makedirs(a.outdir, exist_ok=True)
    with open(os.path.join(a.outdir, "bench_negbin.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
