"""Cholesky + inverse timing at the benchmark size: the single cluster kernel against the panel hybrid (256-wide diagonal blocks on
the cluster kernel, the rest on tcgen05, split over the caller's stream and a side stream), for L = 10 factors and for the 1-2
factors a rank would own if the chain were sharded by factor.  Then the in-kernel clocks of one cluster launch (its phases and
the first 64 x 64 leaf) and the whole call at M = 1024, L = 10, on a dense SPD matrix and on config 2's Kzz.
Usage: python tools/prof_chol.py [M ...]"""
import ctypes, subprocess, sys, torch
sys.path.insert(0, '.')
from gpzoo_b200 import functional as F, _cabi
F.set_sync_checks(False)
torch.manual_seed(0)

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                     capture_output=True, text=True).stdout.strip().splitlines()
name, power, mhz = (s.strip() for s in smi[0].split(",")) if smi else ("?", "?", "0")
print(f"GPU: {name}, power limit {power} W, max SM clock {mhz} MHz (cycles below are converted at that clock)")
us = lambda cyc: cyc / float(mhz) if float(mhz) > 0 else float("nan")


def timeit(fn, n=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def phases(K, thr):
    """Clocks of the first cluster launch (the whole factor on the cluster path, the first 256-wide block on the hybrid)."""
    F.CHOL_TC_MIN_M = thr
    dbg = torch.zeros(10, dtype=torch.int64, device='cuda')
    _cabi.lib().gpz_chol_debug_(ctypes.c_void_p(dbg.data_ptr()))
    F.CholeskyInverse.apply(K)
    torch.cuda.synchronize()
    _cabi.lib().gpz_chol_debug_(ctypes.c_void_p(0))
    c = dbg.cpu().tolist()
    leaf = sum(c[4:10])
    return (f"leaf {us(leaf):.1f} us ({leaf} cycles: load {c[4]} diag0 {c[5]} products {c[6]} diag1 {c[7]} X21 {c[8]} store {c[9]}); "
            f"launch phases: leaf {c[0]} panel {c[1]} trail+leaf {c[2]} inverse {c[3]} = {us(sum(c[:4])):.1f} us")


for M in [int(a) for a in sys.argv[1:]] or [1024]:
    for L in (10, 2, 1):
        Q = torch.randn(L, M, M, device='cuda')
        K = Q @ Q.transpose(1, 2) / M + torch.eye(M, device='cuda')
        ref = torch.linalg.cholesky(K.double())
        out = {}
        for name_, thr in (("cluster", 1 << 30), ("hybrid", 0)):
            F.CHOL_TC_MIN_M = thr
            if name_ == "cluster" and M > 1536:
                continue
            t = timeit(lambda: F.CholeskyInverse.apply(K))
            Lc, Linv = F.CholeskyInverse.apply(K)
            err = float((Lc.double() - ref).norm() / ref.norm())
            erri = float((Linv.double() @ ref - torch.eye(M, device='cuda', dtype=torch.float64)).norm() / M ** 0.5)
            out[name_] = (t, err, erri)
        tt = timeit(lambda: torch.linalg.cholesky(K))
        line = f"M={M} L={L}: " + "  ".join(f"{k} {v[0]:.3f} ms (Lc err {v[1]:.1e}, |Linv Lc - I| {v[2]:.1e})" for k, v in out.items())
        print(line + f"  torch.linalg.cholesky alone {tt:.3f} ms")
        if M <= 1536:
            print(f"  cluster path, L={L}: " + phases(K, 1 << 30))
        print(f"  hybrid, L={L}, first diagonal block: " + phases(K, 0))

# M = 1024, L = 10 on config 2's own Kzz: 1.1 I plus mostly exact zeros and tiny entries (DESIGN §4, "denormals and zero numerators")
from gpzoo_b200 import synthetic
import gpzoo_b200 as gz
pr = synthetic.nsf_problem(N=64, M=1024, L=10, G=4, E=1, seed=1, coord_scale=100.0, lengthscale=1.7, jitter=1e-1, dtype=torch.float32, device='cuda')
kern = gz.kernels.NSF_RBF(L=10)
kern.sigma, kern.lengthscale = torch.nn.Parameter(pr["sigma"]), torch.nn.Parameter(pr["lengthscale"])
with torch.no_grad():
    Kzz = kern(pr["Z"], pr["Z"], _jitter=0.1).contiguous()
Q = torch.randn(10, 1024, 1024, device='cuda')
Kd = Q @ Q.transpose(1, 2) / 1024 + torch.eye(1024, device='cuda')
den = float(((Kzz != 0) & (Kzz.abs() < 1.2e-38)).float().mean())
print(f"config-2 Kzz: fraction of denormal entries {den:.3f}, zeros {float((Kzz == 0).float().mean()):.3f}")
for label, K in (("dense SPD", Kd), ("config-2 Kzz", Kzz)):
    F.CHOL_TC_MIN_M = 0
    t = timeit(lambda: F.CholeskyInverse.apply(K), n=50)
    print(f"M=1024 L=10 {label}: hybrid {t:.3f} ms per call; first diagonal block: " + phases(K, 0))
    F.CHOL_TC_MIN_M = 1 << 30
    print(f"M=1024 L=10 {label}: cluster path {timeit(lambda: F.CholeskyInverse.apply(K)):.3f} ms per call")
