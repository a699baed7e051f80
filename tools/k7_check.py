"""K7 alone: the default fp32 call against the fp64 call on the same inputs, plus its time.
usage: python tools/k7_check.py [G F B E with_lgamma use_idx y_kind]   (y_kind 1 / 2 / 3: counts as uint8 / int16 / int32)"""
import sys, torch
sys.path.insert(0, '.')
from gpzoo_b200 import functional as F

a = [int(x) for x in sys.argv[1:]]
G, Fn, B, E, lg, use_idx, yk = (a + [2000, 10, 32768, 1, 0, 0, 0][len(a):])
YDT = {0: None, 1: torch.uint8, 2: torch.int16, 3: torch.int32}[yk]
torch.manual_seed(0)
dev = 'cuda'
Ntot = B + 1000 if use_idx else B
y = torch.poisson(torch.full((G, Ntot), 0.3, device=dev, dtype=torch.float64))
y[0, :5] = torch.tensor([3., 7., 70., 2., 1.], dtype=torch.float64)
W = torch.rand(G, Fn, device=dev, dtype=torch.float64)
V = 1 + 0.1 * torch.randn(Ntot, device=dev, dtype=torch.float64)
mean = 0.3 * torch.randn(Fn, B, device=dev, dtype=torch.float64)
var = 0.03 + torch.rand(Fn, B, device=dev, dtype=torch.float64)
eps = torch.randn(E, Fn, B, device=dev, dtype=torch.float64)
idx = torch.randperm(Ntot, device=dev)[:B] if use_idx else None


def run(dt):
    leaves = [t.to(dt).clone().requires_grad_(True) for t in (W, V, mean, var)]
    ll = F.PoissonLL.apply(y.to(YDT if (YDT is not None and dt == torch.float32) else dt), idx, leaves[0], leaves[1], leaves[2], leaves[3], eps.to(dt), Fn, 5e-2, True, bool(lg))
    ll.backward()
    return ll.detach().double(), [t.grad.double() for t in leaves]


ref, gref = run(torch.float64)
out, gout = run(torch.float32)
rel = lambda x, r: float((x - r).norm() / r.norm())
print(f"G={G} F={Fn} B={B} E={E} lgamma={lg} idx={use_idx}: ll {float(out):.6f} ref {float(ref):.6f} rel {rel(out, ref):.2e}  "
      + "  ".join(f"d{n} {rel(g, r):.2e}" for n, g, r in zip(("W", "V", "mean", "var"), gout, gref)))
y32, W32, V32, m32, v32, e32 = (t.float() for t in (y, W, V, mean, var, eps))
if YDT is not None:
    y32 = y32.to(YDT)
for _ in range(4):
    F.PoissonLL.apply(y32, idx, W32, V32, m32, v32, e32, Fn, 5e-2, True, bool(lg))
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(20):
    F.PoissonLL.apply(y32, idx, W32, V32, m32, v32, e32, Fn, 5e-2, True, bool(lg))
e1.record(); torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / 20
print(f"  {ms:.4f} ms per call (3 launches), {y32.element_size() * G * B * E / ms / 1e6:.0f} GB/s of y ({y32.dtype})")
