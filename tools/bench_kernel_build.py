"""K1 per covariance kind: the split-FP16 forward (gpz_kernel_build_fwd_h_f32), the fp32 backward (gpz_kernel_build_bwd_f32)
and the whole model step, for kind 0 (RBF), 1 (Matern-3/2), 2 (Matern-1/2) and 3 (Matern-5/2).

    python tools/bench_kernel_build.py OUTDIR [--reps 200] [--warmup 20] [--step-reps 100]

Workloads, at config 2's shape (L = 10, M = 1024 inducing points, N = 32768 spots, D = 2, fp32):
  * each kernel call alone: milliseconds per call (CUDA events over --reps launches after --warmup, the four kinds alternated
    in three rounds, median of the rounds).  The forward writes and the backward reads 4 bytes per entry (1.34 GB per call,
    ten times the 126 MB L2); the buffers are replicated until the copies exceed 256 MB and the launches cycle through them,
    so no call is served from L2.  GB/s counts those 4 L M N bytes and is also given as a fraction of 6538 GB/s, the copy
    bandwidth DESIGN.md section 4 uses;
  * one config-2 NSF2(SVGP(kernel)).elbo fwd + bwd step per kind (batched_RBF / batched_Matern32 / 12 / 52 with (L,)
    parameters, same inducing points, variational parameters and counts), alternated the same way (--step-reps steps per round).
Every round's time is recorded next to the median, so the spread can be read off.
The GPU's name and power limit are read with nvidia-smi in the same run.  Writes OUTDIR/bench_kernel_build.json.
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
COPY_GBS = 6538.0                     # DESIGN.md section 4: the measured HBM copy bandwidth its fractions of peak use
KINDS = {0: "batched_RBF", 1: "batched_Matern32", 2: "batched_Matern12", 3: "batched_Matern52"}
L, M, N, D = 10, 1024, 32768, 2


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


def _summary(rounds_ms, nbytes):
    ms = statistics.median(rounds_ms)
    gbs = nbytes / (ms * 1e-3) / 1e9
    return dict(ms=ms, gb_per_s=gbs, fraction_of_copy=gbs / COPY_GBS, rounds_ms=rounds_ms)


def call_points(reps, warmup, seed=0):
    import torch
    from gpzoo_b200 import synthetic
    from gpzoo_b200._cabi import call
    dt, dev = torch.float32, "cuda"
    prob = synthetic.nsf_problem(N=N, M=M, L=L, G=8, E=1, seed=seed, coord_scale=100.0, lengthscale=1.7, jitter=0.1,
                                 dtype=dt, device=dev)
    Z, X = prob["Z"].contiguous(), prob["X"].contiguous()
    sigma, ls = prob["sigma"].reshape(-1).contiguous(), prob["lengthscale"].reshape(-1).contiguous()
    nbytes = 4 * L * M * N
    copies = max(1, math.ceil(L2_DEFEAT_BYTES / nbytes))
    planes = [torch.empty((2, L, M, N), dtype=torch.float16, device=dev) for _ in range(copies)]
    sK = torch.empty(L, dtype=dt, device=dev)
    g = torch.Generator(device=dev).manual_seed(seed + 1)
    Gs = [torch.randn(L, M, N, generator=g, device=dev) for _ in range(copies)]
    g_x1, g_x2 = torch.empty_like(Z), torch.empty_like(X)
    g_s, g_l = torch.empty_like(sigma), torch.empty_like(ls)
    ws = torch.empty(3 * L + M * D, dtype=torch.float64, device=dev)

    def fwd(kind):
        def f(i):
            p = planes[i % copies]
            call("kernel_build_fwd_h", dt, Z, X, sigma, ls, None, None, None, None, M, N, D, L, 0, kind, 1.0, 0.0, p[0], p[1], sK)
        return f

    def bwd(kind):
        def f(i):
            call("kernel_build_bwd", dt, Z, X, sigma, ls, None, None, None, None, M, N, D, L, 0, kind, 1.0, Gs[i % copies],
                 g_x1, g_x2, g_s, g_l, None, ws)
        return f
    tf = _time({k: fwd(k) for k in KINDS}, reps, warmup)
    tb = _time({k: bwd(k) for k in KINDS}, reps, warmup)
    out = {}
    for k, name in KINDS.items():
        out[name] = dict(kind=k, fwd_h=_summary(tf[k], nbytes), bwd=_summary(tb[k], nbytes))
        out[name]["fwd_h"]["vs_rbf"] = out[name]["fwd_h"]["ms"] / statistics.median(tf[0])
        out[name]["bwd"]["vs_rbf"] = out[name]["bwd"]["ms"] / statistics.median(tb[0])
    return dict(buffer_copies=copies, bytes_per_call=nbytes, kinds=out)


def step_points(reps, warmup):
    """config 2 (bench.py's problem): one NSF2(SVGP(kernel)).elbo fwd+bwd per kind, same parameters and counts."""
    import torch
    import gpzoo_b200 as gz
    from gpzoo_b200 import synthetic
    prob = synthetic.nsf_problem(N=N, M=M, L=L, G=2000, E=1, seed=0, coord_scale=100.0, lengthscale=1.7, jitter=0.1,
                                 dtype=torch.float32, device="cuda")
    models = {}
    for k, name in KINDS.items():
        kern = getattr(gz.kernels, name)()
        kern.sigma = torch.nn.Parameter(prob["sigma"].reshape(-1).clone())
        kern.lengthscale = torch.nn.Parameter(prob["lengthscale"].reshape(-1).clone())
        gp = gz.gp.SVGP(kern, dim=2, M=M, jitter=prob["jitter"])
        gp.Z, gp.mu, gp.Lu = (torch.nn.Parameter(prob[key].clone()) for key in ("Z", "mu", "Lu_raw"))
        m = gz.likelihoods.NSF2(gp, prob["y"], L=L).cuda()
        m.W, m.V = torch.nn.Parameter(prob["W"].clone()), torch.nn.Parameter(prob["V"].clone())
        models[k] = m
    X, y = prob["X"], prob["y"]
    eps = torch.randn(1, L, N, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))

    def step(m):
        def f(i):
            m.zero_grad(set_to_none=True)
            m.elbo(X, y, E=1, eps=eps).backward()
        return f
    gz.functional.set_sync_checks(False)
    t = _time({k: step(m) for k, m in models.items()}, reps, warmup)
    rbf = statistics.median(t[0])
    return {name: dict(kind=k, step_ms=statistics.median(t[k]), vs_rbf=statistics.median(t[k]) / rbf, rounds_ms=t[k])
            for k, name in KINDS.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--step-reps", type=int, default=100)      # 100 steps of ~8 ms: a window of 0.8 s per round
    a = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "bench_kernel_build.py measures on a CUDA device"
    res = dict(gpu_info(), shape=dict(L=L, M=M, N=N, D=D, dtype="float32"), copy_gb_per_s=COPY_GBS)
    with torch.no_grad():
        res["calls"] = call_points(a.reps, a.warmup)
    res["step"] = step_points(a.step_reps, 5)
    os.makedirs(a.outdir, exist_ok=True)
    with open(os.path.join(a.outdir, "bench_kernel_build.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
