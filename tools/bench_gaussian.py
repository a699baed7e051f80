"""K7-G against K7: the fused Gaussian factor-model call (gpz_gaussian_fwdbwd_f32) and the dense Poisson call on the same shape.

    python tools/bench_gaussian.py OUTDIR [--reps 200] [--warmup 20] [--step-reps 200]

Workloads, at config 2's shape (G = 2000, B = 32768, F = 10, fp32; the Poisson call with E = 1):
  * the likelihood call alone: milliseconds per call (CUDA events over --reps launches after --warmup, Gaussian and Poisson
    alternated in three rounds, median of the rounds).  y is replicated until the copies exceed 256 MB and the launches cycle
    through them, so no call reads y from the 126 MB L2.  The y bytes read per call over the time give the achieved read rate;
  * one full config-2 model.elbo fwd+bwd step of RSF(SVGP) against NSF2(SVGP) (same GP parameters and loadings, y the same fp32
    matrix), alternated the same way (--step-reps steps per round).
Every round's time is recorded next to the median, so the spread can be read off.
The GPU's name and power limit are read with nvidia-smi in the same run.  Writes OUTDIR/bench_gaussian.json.
"""
import argparse
import json
import math
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.bench_negbin import L2_DEFEAT_BYTES, _time, gpu_info  # noqa: E402


def call_point(reps, warmup, G=2000, B=32768, F=10, seed=0):
    import torch
    from gpzoo_b200 import functional as Fn
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(seed)
    y = 2 * torch.randn(G, B, generator=g, device=dev)
    counts = torch.poisson(2 * torch.rand(G, B, generator=g, device=dev))
    copies = max(1, math.ceil(L2_DEFEAT_BYTES / (y.numel() * y.element_size())))
    ys = [y] + [y.clone() for _ in range(copies - 1)]
    cs = [counts] + [counts.clone() for _ in range(copies - 1)]
    W = torch.randn(G, F, generator=g, device=dev)
    bias, noise = torch.randn(G, generator=g, device=dev), torch.randn(G, generator=g, device=dev)
    V = 1 + 0.2 * torch.randn(B, generator=g, device=dev)
    mean = 0.3 * torch.randn(F, B, generator=g, device=dev)
    var = 0.05 + 0.3 * torch.rand(F, B, generator=g, device=dev)
    eps = torch.randn(1, F, B, generator=g, device=dev)
    ga = lambda i: Fn.GaussianLL.apply(ys[i % copies], None, W, bias, noise, mean, var, F, 5e-2)
    po = lambda i: Fn.PoissonLL.apply(cs[i % copies], None, W - 1.0, V, mean, var, eps, F, 5e-2, True, True)
    with torch.no_grad():
        t = _time(dict(gaussian=ga, poisson=po), reps, warmup)
    ga, po = statistics.median(t["gaussian"]), statistics.median(t["poisson"])
    y_bytes = y.numel() * y.element_size()
    return dict(y_copies=copies, y_bytes=y_bytes, gaussian_ms=ga, poisson_ms=po, ratio=ga / po,
                gaussian_y_read_GBps=y_bytes / (ga * 1e-3) / 1e9, gaussian_rounds_ms=t["gaussian"], poisson_rounds_ms=t["poisson"])


def step_point(reps, warmup):
    """config 2 (bench.py's problem): one RSF and one NSF2 elbo fwd+bwd over the same SVGP parameters and loadings."""
    import torch
    import gpzoo_b200 as gz
    from gpzoo_b200 import synthetic
    prob = synthetic.nsf_problem(N=32768, M=1024, L=10, G=2000, E=1, seed=0, coord_scale=100.0, lengthscale=1.7, jitter=0.1,
                                 dtype=torch.float32, device="cuda")
    models = {}
    for name, cls in (("rsf", gz.likelihoods.RSF), ("nsf2", gz.likelihoods.NSF2)):
        kern = gz.kernels.NSF_RBF(L=10)
        kern.sigma, kern.lengthscale = torch.nn.Parameter(prob["sigma"].clone()), torch.nn.Parameter(prob["lengthscale"].clone())
        gp = gz.gp.SVGP(kern, dim=2, M=1024, jitter=prob["jitter"])
        gp.Z, gp.mu, gp.Lu = (torch.nn.Parameter(prob[k].clone()) for k in ("Z", "mu", "Lu_raw"))
        m = cls(gp, prob["y"], L=10).cuda()
        m.W = torch.nn.Parameter(prob["W"].clone())
        if name == "nsf2":
            m.V = torch.nn.Parameter(prob["V"].clone())
        models[name] = m
    X, y = prob["X"], prob["y"].float()
    eps = torch.randn(1, 10, 32768, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))

    def step(m):
        def f(i):
            m.zero_grad(set_to_none=True)
            m.elbo(X, y, E=1, eps=eps).backward()
        return f
    gz.functional.set_sync_checks(False)
    t = _time({k: step(m) for k, m in models.items()}, reps, warmup)
    rs, ns = statistics.median(t["rsf"]), statistics.median(t["nsf2"])
    return dict(rsf_step_ms=rs, nsf2_step_ms=ns, ratio=rs / ns, rsf_rounds_ms=t["rsf"], nsf2_rounds_ms=t["nsf2"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--step-reps", type=int, default=200)      # 200 steps of ~8 ms: a window of 1.6 s per round
    a = ap.parse_args()
    res = dict(gpu_info(), shape=dict(G=2000, B=32768, F=10, dtype="float32"))
    res["call"] = call_point(a.reps, a.warmup)
    res["step"] = step_point(a.step_reps, 5)
    os.makedirs(a.outdir, exist_ok=True)
    with open(os.path.join(a.outdir, "bench_gaussian.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
