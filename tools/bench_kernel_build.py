"""K1 per covariance kind: the split-FP16 forward (gpz_kernel_build_fwd_h_f32), the fp32 backward (gpz_kernel_build_bwd_f32)
and the whole model step, for kind 0 (RBF), 1 (Matern-3/2), 2 (Matern-1/2) and 3 (Matern-5/2), each isotropic and with
per-dimension (ARD) lengthscales (gpz_kernel_build_ard_fwd_h_f32 / gpz_kernel_build_ard_bwd_f32).

    python tools/bench_kernel_build.py OUTDIR [--reps 200] [--warmup 20] [--step-reps 100]

Workloads, at config 2's shape (L = 10, M = 1024 inducing points, N = 32768 spots, fp32), for D = 2 (config 2's) and D = 3:
  * each kernel call alone: milliseconds per call (CUDA events over --reps launches after --warmup, the eight variants (four
    kinds, isotropic and ARD) alternated in three rounds, median of the rounds).  The forward writes and the backward reads 4 bytes per entry (1.34 GB per call,
    ten times the 126 MB L2); the buffers are replicated until the copies exceed 256 MB and the launches cycle through them,
    so no call is served from L2.  GB/s counts those 4 L M N bytes and is also given as a fraction of 6538 GB/s, the copy
    bandwidth DESIGN.md section 4 uses;
  * one config-2 NSF2(SVGP(kernel)).elbo fwd + bwd step per variant (batched_RBF / batched_Matern32 / 12 / 52 with (L,)
    parameters, batched_ARD_* with (L,) sigma and (L, D) lengthscales; same inducing points, variational parameters and
    counts), alternated the same way (--step-reps steps per round).
The ARD lengthscales are the isotropic ones times (2, 1/2) for D = 2 and (2, 1, 1/2) for D = 3 (a ratio of 4 between axes,
geometric mean 1).  ARD rows carry vs_isotropic, the ratio to the isotropic row of the same kind and D.
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
ARD_KINDS = {0: "batched_ARD_RBF", 1: "batched_ARD_Matern32", 2: "batched_ARD_Matern12", 3: "batched_ARD_Matern52"}
VARIANTS = [(k, ard) for k in KINDS for ard in (False, True)]
L, M, N = 10, 1024, 32768
DIMS = (2, 3)


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


def _name(kind, ard):
    return (ARD_KINDS if ard else KINDS)[kind]


def _ard_ls(ls, D):
    """(L,) isotropic lengthscales -> (L, D): times (2, 1/2) or (2, 1, 1/2)."""
    import torch
    axes = torch.tensor([2.0, 0.5] if D == 2 else [2.0, 1.0, 0.5], dtype=ls.dtype, device=ls.device)
    return (ls.reshape(-1, 1) * axes).contiguous()


def _with_ratios(out, times, key):
    """vs_rbf on the isotropic rows, vs_isotropic on the ARD rows."""
    for (k, ard), t in times.items():
        ref = times[(k, False)] if ard else times[(0, False)]
        out[_name(k, ard)][key]["vs_isotropic" if ard else "vs_rbf"] = statistics.median(t) / statistics.median(ref)


def call_points(reps, warmup, D, seed=0):
    import torch
    from gpzoo_b200 import synthetic
    from gpzoo_b200._cabi import call
    dt, dev = torch.float32, "cuda"
    prob = synthetic.nsf_problem(N=N, M=M, L=L, G=8, D=D, E=1, seed=seed, coord_scale=100.0, lengthscale=1.7, jitter=0.1,
                                 dtype=dt, device=dev)
    Z, X = prob["Z"].contiguous(), prob["X"].contiguous()
    sigma, ls = prob["sigma"].reshape(-1).contiguous(), prob["lengthscale"].reshape(-1).contiguous()
    ls_ard = _ard_ls(ls, D)
    nbytes = 4 * L * M * N
    copies = max(1, math.ceil(L2_DEFEAT_BYTES / nbytes))
    planes = [torch.empty((2, L, M, N), dtype=torch.float16, device=dev) for _ in range(copies)]
    sK = torch.empty(L, dtype=dt, device=dev)
    g = torch.Generator(device=dev).manual_seed(seed + 1)
    Gs = [torch.randn(L, M, N, generator=g, device=dev) for _ in range(copies)]
    g_x1, g_x2 = torch.empty_like(Z), torch.empty_like(X)
    g_s, g_l, g_la = torch.empty_like(sigma), torch.empty_like(ls), torch.empty_like(ls_ard)
    ws = torch.empty(L + L * D + M * D + 2 * L, dtype=torch.float64, device=dev)       # either call's workspace

    def fwd(kind, ard):
        def f(i):
            p = planes[i % copies]
            if ard:
                call("kernel_build_ard_fwd_h", dt, Z, X, sigma, ls_ard, M, N, D, L, kind, 0.0, p[0], p[1], sK)
            else:
                call("kernel_build_fwd_h", dt, Z, X, sigma, ls, None, None, None, None, M, N, D, L, 0, kind, 1.0, 0.0, p[0], p[1],
                     sK)
        return f

    def bwd(kind, ard):
        def f(i):
            if ard:
                call("kernel_build_ard_bwd", dt, Z, X, sigma, ls_ard, M, N, D, L, kind, Gs[i % copies], g_x1, g_x2, g_s, g_la, ws)
            else:
                call("kernel_build_bwd", dt, Z, X, sigma, ls, None, None, None, None, M, N, D, L, 0, kind, 1.0, Gs[i % copies],
                     g_x1, g_x2, g_s, g_l, None, ws)
        return f
    tf = _time({v: fwd(*v) for v in VARIANTS}, reps, warmup)
    tb = _time({v: bwd(*v) for v in VARIANTS}, reps, warmup)
    out = {_name(k, ard): dict(kind=k, ard=ard, fwd_h=_summary(tf[(k, ard)], nbytes), bwd=_summary(tb[(k, ard)], nbytes))
           for k, ard in VARIANTS}
    _with_ratios(out, tf, "fwd_h")
    _with_ratios(out, tb, "bwd")
    return dict(buffer_copies=copies, bytes_per_call=nbytes, kinds=out)


def step_points(reps, warmup, D):
    """config 2 (bench.py's problem, D = 2, and the same at D = 3): one NSF2(SVGP(kernel)).elbo fwd+bwd per variant, same
    parameters and counts."""
    import torch
    import gpzoo_b200 as gz
    from gpzoo_b200 import synthetic
    prob = synthetic.nsf_problem(N=N, M=M, L=L, G=2000, D=D, E=1, seed=0, coord_scale=100.0, lengthscale=1.7, jitter=0.1,
                                 dtype=torch.float32, device="cuda")
    models = {}
    for k, ard in VARIANTS:
        kern = getattr(gz.kernels, _name(k, ard))(dim=D) if ard else getattr(gz.kernels, _name(k, ard))()
        kern.sigma = torch.nn.Parameter(prob["sigma"].reshape(-1).clone())
        ls = prob["lengthscale"].reshape(-1)
        kern.lengthscale = torch.nn.Parameter(_ard_ls(ls, D) if ard else ls.clone())
        gp = gz.gp.SVGP(kern, dim=D, M=M, jitter=prob["jitter"])
        gp.Z, gp.mu, gp.Lu = (torch.nn.Parameter(prob[key].clone()) for key in ("Z", "mu", "Lu_raw"))
        m = gz.likelihoods.NSF2(gp, prob["y"], L=L).cuda()
        m.W, m.V = torch.nn.Parameter(prob["W"].clone()), torch.nn.Parameter(prob["V"].clone())
        models[(k, ard)] = m
    X, y = prob["X"], prob["y"]
    eps = torch.randn(1, L, N, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))

    def step(m):
        def f(i):
            m.zero_grad(set_to_none=True)
            m.elbo(X, y, E=1, eps=eps).backward()
        return f
    gz.functional.set_sync_checks(False)
    t = _time({v: step(m) for v, m in models.items()}, reps, warmup)
    out = {_name(k, ard): dict(kind=k, ard=ard, step=dict(ms=statistics.median(t[(k, ard)]), rounds_ms=t[(k, ard)]))
           for k, ard in VARIANTS}
    _with_ratios(out, t, "step")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--step-reps", type=int, default=100)      # 100 steps of ~8 ms: a window of 0.8 s per round
    a = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "bench_kernel_build.py measures on a CUDA device"
    res = dict(gpu_info(), shape=dict(L=L, M=M, N=N, D=list(DIMS), dtype="float32"), copy_gb_per_s=COPY_GBS)
    for D in DIMS:
        with torch.no_grad():
            res[f"calls_D{D}"] = call_points(a.reps, a.warmup, D)
        torch.cuda.empty_cache()
        res[f"step_D{D}"] = step_points(a.step_reps, 5, D)
        torch.cuda.empty_cache()
    os.makedirs(a.outdir, exist_ok=True)
    with open(os.path.join(a.outdir, "bench_kernel_build.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
