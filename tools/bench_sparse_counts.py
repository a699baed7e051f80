"""K7 on sparse counts: the CSC call (SparseCounts -> gpz_poisson_fwdbwd_csc_f32) against the dense K7 call with fp32 and uint8 y.

    python tools/bench_sparse_counts.py OUTDIR [--reps 200] [--warmup 20]

Workloads
  * config 2's shape (G = 2000, B = 32768, F = 10, E = 1) on the benchmark's synthetic counts (bench.make_problem, 26.3 % nonzero)
    and on the same counts thinned by a seeded Bernoulli mask to 10 %, 3 % and 1 %;
  * G = 17702, N = 39694 (the Slide-seq V2 matrix of SURVEY.md §4) at 3 % and 1 %, synthetic counts;
  * one full config-2 model.elbo fwd+bwd step with dense and with sparse y.
Each K7 point: milliseconds per call (CUDA events over --reps launches after --warmup, the variants alternated in three rounds,
median of the rounds), the bytes of y, and the agreement of ll and of the four gradients between the dense fp32 and the CSC call.
Every input array is replicated until the copies exceed 256 MB and the launches cycle through them, so no call reads y from the
126 MB L2.  The GPU's name and power limit are read with nvidia-smi in the same run.  Writes OUTDIR/bench_sparse_counts.json.
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


def relerr(a, b):
    a, b = a.detach().double().reshape(-1), b.detach().double().reshape(-1)
    n = float(b.norm())
    return float((a - b).norm()) / n if n > 0 else float((a - b).norm())


def thin(y, density, seed):
    """Keep each nonzero of y with probability density / (current density) (seeded Bernoulli mask)."""
    import torch
    cur = float((y != 0).float().mean())
    if density >= cur:
        return y
    g = torch.Generator(device=y.device).manual_seed(seed)
    return y * (torch.rand(y.shape, generator=g, device=y.device) < density / cur)


def k7_point(label, y, F, E, reps, warmup, seed=0):
    """Time dense fp32 / dense uint8 / CSC PoissonLL calls on the same G x N counts y (fp32, on the device)."""
    import torch
    from gpzoo_b200 import SparseCounts, functional as Fn
    dev = y.device
    G, N = y.shape
    g = torch.Generator(device=dev).manual_seed(seed)
    W = torch.rand(G, F, generator=g, device=dev) - 1.0
    V = 1 + 0.2 * torch.randn(N, generator=g, device=dev)
    mean = 0.3 * torch.randn(F, N, generator=g, device=dev)
    spread = 0.05 + 0.3 * torch.rand(F, N, generator=g, device=dev)
    eps = torch.randn(E, F, N, generator=g, device=dev)
    ys = SparseCounts.from_dense(y)
    variants = dict(dense_f32=y, dense_u8=y.to(torch.uint8), csc=ys)
    nbytes = dict(dense_f32=y.numel() * 4, dense_u8=y.numel(),
                  csc=ys.indptr.numel() * 8 + ys.nnz * (4 + ys.values.element_size()))

    def call(yy, grads=False):
        lv = [t.clone().requires_grad_(grads) for t in (W, V, mean, spread)]
        out = Fn.PoissonLL.apply(yy, None, lv[0], lv[1], lv[2], lv[3], eps, F, 5e-2, True, True)
        if grads:
            out.backward()
            return out.detach(), [t.grad for t in lv]
        return out

    o_d, g_d = call(y, True)
    res = {}
    for k in ("dense_u8", "csc"):
        o, gr = call(variants[k], True)
        res[k] = dict(ll_rel=relerr(o, o_d), **{"g%s_rel" % n: relerr(a, b) for n, a, b in zip(("W", "V", "mean", "spread"), gr, g_d)})
    del o_d, g_d
    copies = {}
    for k, v in variants.items():
        n = max(1, min(128, math.ceil(L2_DEFEAT_BYTES / nbytes[k])))
        if k == "csc":
            copies[k] = [v] + [SparseCounts(v.indptr.clone(), v.genes.clone(), v.values.clone(), v.n_genes) for _ in range(n - 1)]
        else:
            copies[k] = [v] + [v.clone() for _ in range(n - 1)]
    times = {k: [] for k in variants}
    with torch.no_grad():
        for k in variants:
            for i in range(warmup):
                call(copies[k][i % len(copies[k])])
        torch.cuda.synchronize()
        for _ in range(3):
            for k in variants:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for i in range(reps):
                    call(copies[k][i % len(copies[k])])
                e1.record()
                torch.cuda.synchronize()
                times[k].append(e0.elapsed_time(e1) / reps)
    del copies
    torch.cuda.empty_cache()
    pt = dict(point=label, G=G, N=N, F=F, E=E, nnz=ys.nnz, density=ys.nnz / (G * N), reps=reps,
              ms={k: statistics.median(v) for k, v in times.items()}, ms_rounds=times, y_bytes=nbytes,
              agreement_vs_dense_f32=res)
    print(json.dumps(pt), flush=True)
    return pt


def elbo_step_point(reps, warmup):
    """One config-2 model.elbo fwd+bwd step, dense fp32 y against SparseCounts y (alternated, three rounds)."""
    import torch
    import bench
    from gpzoo_b200 import SparseCounts, functional
    functional.set_sync_checks(False)
    c = bench.CONFIGS[2]
    dev = torch.device("cuda")
    prob = bench.make_problem(c, c["N"], c["seed"], torch.float32)
    model, _ = bench.build_model(c, prob, torch.float32, dev)
    X, eps = prob["X"].to(dev), prob["eps"].to(dev)
    ys = dict(dense_f32=prob["y"].to(dev), csc=SparseCounts.from_dense(prob["y"]).to(dev))

    def step(y):
        for p in model.parameters():
            p.grad = None
        elbo = model.elbo(X, y, E=c["E"], eps=eps)
        (-elbo).backward()
        return elbo.detach()

    e_d, e_s = step(ys["dense_f32"]), step(ys["csc"])
    times = {k: [] for k in ys}
    for k in ys:
        for _ in range(warmup):
            step(ys[k])
    torch.cuda.synchronize()
    for _ in range(3):
        for k in ys:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                step(ys[k])
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1) / reps)
    functional.check_cholesky_info()
    pt = dict(point="config2 model.elbo fwd+bwd step", reps=reps, ms={k: statistics.median(v) for k, v in times.items()},
              ms_rounds=times, elbo_rel=relerr(e_s, e_d))
    print(json.dumps(pt), flush=True)
    return pt


def crossover(points, a="csc", b="dense_u8"):
    """Density at which the CSC call and the dense uint8 call take the same time (linear interpolation between measured points)."""
    pts = sorted((p["density"], p["ms"][a] - p["ms"][b]) for p in points)
    for (d0, x0), (d1, x1) in zip(pts, pts[1:]):
        if x0 <= 0 < x1 or x0 >= 0 > x1:
            return d0 + (d1 - d0) * (0 - x0) / (x1 - x0)
    return None


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("outdir")
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--step-reps", type=int, default=50)
    args = ap.parse_args()
    import torch
    import bench
    from gpzoo_b200 import _cabi
    if not torch.cuda.is_available():
        raise SystemExit("bench_sparse_counts needs a CUDA device")
    _cabi.lib()
    os.makedirs(args.outdir, exist_ok=True)
    info = gpu_info()
    print(json.dumps(info), flush=True)
    dev = torch.device("cuda")
    c = bench.CONFIGS[2]
    y0 = bench.make_problem(c, c["N"], c["seed"], torch.float32)["y"].to(dev)
    cfg2 = []
    for d in (None, 0.10, 0.03, 0.01):
        y = y0 if d is None else thin(y0, d, seed=11)
        cfg2.append(k7_point("config2 shape, %s" % ("synthetic density" if d is None else "thinned to %g" % d), y, 10, 1,
                             args.reps, args.warmup))
        del y
    del y0
    big = []
    G, N = 17702, 39694
    for d in (0.03, 0.01):
        g = torch.Generator(device=dev).manual_seed(12)
        y = (torch.rand(G, N, generator=g, device=dev) < d) * (1 + torch.poisson(torch.full((G, N), 0.5, device=dev), generator=g))
        big.append(k7_point("G=17702 N=39694 at %g" % d, y.float(), 10, 1, max(20, args.reps // 4), args.warmup))
        del y
        torch.cuda.empty_cache()
    step = elbo_step_point(args.step_reps, 5)
    out = dict(info, config2=cfg2, slideseq_v2_shape=big, elbo_step=step, crossover_density_vs_dense_u8_config2=crossover(cfg2),
               crossover_density_vs_dense_f32_config2=crossover(cfg2, b="dense_f32"))
    with open(os.path.join(args.outdir, "bench_sparse_counts.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(dict(info, crossover_u8=out["crossover_density_vs_dense_u8_config2"],
                          crossover_f32=out["crossover_density_vs_dense_f32_config2"])))


if __name__ == "__main__":
    main()
