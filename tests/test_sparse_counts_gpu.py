"""GPU: the fused Poisson ELBO on sparse counts (SparseCounts -> gpz_poisson_fwdbwd_csc_*) against the CPU oracle, against the
dense K7 call on the same inputs, at edge cases of the format and of the kernel's two d/dW paths, and through the models."""
import copy

import pytest
import torch

from gpzoo_b200.counts import SparseCounts
from tests.helpers import load_golden, relerr

pytestmark = pytest.mark.gpu
DEV = "cuda"
KINDS = (None, torch.uint8, torch.int16, torch.int32)       # None: values in the compute type


def _with_kind(s, kind, dt):
    """The same counts with the values stored as `kind` (None -> dt)."""
    return SparseCounts(s.indptr, s.genes, s.values.to(kind or dt), s.n_genes)


def _problem(G, Fn, Ntot, E, B=None, seed=0, density=0.3, nvar=None, scale=2.0):
    g = torch.Generator().manual_seed(seed)
    y = torch.poisson(torch.rand(G, Ntot, generator=g, dtype=torch.float64) * scale, generator=g)
    y = y * (torch.rand(G, Ntot, generator=g, dtype=torch.float64) < density)
    idx = None if B is None else torch.randperm(Ntot, generator=g)[:B]
    B = Ntot if idx is None else B
    p = dict(y=y, idx=idx, W=torch.rand(G, Fn, generator=g, dtype=torch.float64),
             V=1 + 0.2 * torch.randn(Ntot, generator=g, dtype=torch.float64),
             mean=0.3 * torch.randn(Fn, B, generator=g, dtype=torch.float64),
             spread=0.05 + 0.3 * torch.rand(Fn, B, generator=g, dtype=torch.float64),
             eps=torch.randn(E, Fn, B, generator=g, dtype=torch.float64), nvar=Fn // 2 if nvar is None else nvar)
    p["spread"][0, :7] = 1e-3                              # exercise the variance clamp (5e-2)
    return p


def _oracle(p, soft=True, with_lgamma=True):
    from oracle import gpzoo_oracle as O
    leaves = [p[k].clone().requires_grad_(True) for k in ("W", "V", "mean", "spread")]
    Wl, Vl, ml, sl = leaves
    nv = p["nvar"]
    sd = torch.cat((torch.clamp(sl[:nv], min=5e-2).sqrt(), sl[nv:]), 0)
    rate = O.poisson_rate(Wl, ml + p["eps"] * sd, Vl if p["idx"] is None else Vl[p["idx"]], softplus_W=soft)
    ll = O.poisson_loglik(p["y"] if p["idx"] is None else p["y"][:, p["idx"]], rate, with_lgamma=with_lgamma)
    ll.backward()
    return ll.detach(), [t.grad for t in leaves]


def _run(p, y, dt, soft=True, with_lgamma=True):
    """PoissonLL on the device with y dense or sparse; returns ll, the four gradients and the C-ABI calls made."""
    from gpzoo_b200 import _cabi, functional as F
    lv = [p[k].to(DEV, dt).requires_grad_(True) for k in ("W", "V", "mean", "spread")]
    idx = None if p["idx"] is None else p["idx"].to(DEV)
    _cabi.profile = {}
    try:
        out = F.PoissonLL.apply(y, idx, lv[0], lv[1], lv[2], lv[3], p["eps"].to(DEV, dt), p["nvar"], 5e-2, soft, with_lgamma)
    finally:
        calls, _cabi.profile = set(_cabi.profile), None
    out.backward()
    return out.detach(), [t.grad for t in lv], calls


CASES = dict(full=dict(G=45, Fn=5, Ntot=300, E=1), idx=dict(G=45, Fn=5, Ntot=300, E=2, B=170),
             hybrid_raw=dict(G=45, Fn=5, Ntot=300, E=1), F20=dict(G=60, Fn=20, Ntot=257, E=1, nvar=10),
             E3=dict(G=45, Fn=7, Ntot=300, E=3, B=211))


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("case", list(CASES))
def test_csc_vs_oracle(dt, case):
    p = _problem(seed=3, **CASES[case])
    p["y"][5] = 0                                          # an empty gene
    p["y"][:, 11] = 0                                      # an empty spot
    soft = case != "hybrid_raw"
    ll_r, g_r = _oracle(p, soft)
    s = SparseCounts.from_dense(p["y"]).to(DEV)
    tol = 1e-11 if dt == torch.float64 else 3e-5
    for kind in KINDS:
        out, grads, calls = _run(p, _with_kind(s, kind, dt), dt, soft)
        assert "poisson_fwdbwd_csc" in calls and "poisson_fwdbwd" not in calls, calls
        assert relerr(out, ll_r) < tol, (kind, relerr(out, ll_r))
        for name, a, b in zip(("W", "V", "mean", "spread"), grads, g_r):
            assert relerr(a, b) < tol, (kind, name, relerr(a, b))


@pytest.mark.parametrize("case", ["full", "idx", "hybrid_raw"])
def test_csc_vs_dense_fp32(case):
    """Same inputs, dense y (K7) and sparse y (K7-CSC), fp32: ll within 1e-6, gradients within 1e-5."""
    p = _problem(G=300, Fn=10, Ntot=3000, E=1, B=2001 if case == "idx" else None, seed=4, density=0.1)
    soft = case != "hybrid_raw"
    o_d, g_d, _ = _run(p, p["y"].to(DEV, torch.float32), torch.float32, soft)
    o_s, g_s, _ = _run(p, SparseCounts.from_dense(p["y"]).to(DEV), torch.float32, soft)
    assert relerr(o_s, o_d) < 1e-6
    for name, a, b in zip(("W", "V", "mean", "spread"), g_s, g_d):
        assert relerr(a, b) < 1e-5, (name, relerr(a, b))


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
def test_csc_edge_cases(dt):
    tol = 1e-11 if dt == torch.float64 else 3e-5
    # nnz = 0: only the closed-form -rate terms
    p = _problem(G=30, Fn=4, Ntot=100, E=2, seed=5, density=0.0)
    s = SparseCounts.from_dense(p["y"]).to(DEV)
    assert s.nnz == 0
    ll_r, g_r = _oracle(p)
    out, grads, _ = _run(p, s, dt)
    assert relerr(out, ll_r) < tol and all(relerr(a, b) < tol for a, b in zip(grads, g_r))
    # one spot holding all G genes among empty spots; B (through idx) not a multiple of the warps of a CTA
    p = _problem(G=2000, Fn=6, Ntot=1200, E=1, B=1001, seed=6, density=0.002, scale=3.0)
    p["y"][:, p["idx"][17]] = 1 + torch.arange(2000, dtype=torch.float64) % 5
    ll_r, g_r = _oracle(p)
    out, grads, _ = _run(p, SparseCounts.from_dense(p["y"]).to(DEV), dt)
    assert relerr(out, ll_r) < tol and all(relerr(a, b) < tol for a, b in zip(grads, g_r))


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
def test_csc_large_gene_count(dt):
    """G F beyond the per-CTA shared-memory accumulator (G = 20000, F = 10): the global-accumulator path."""
    from gpzoo_b200 import _cabi
    assert _cabi.lib().gpz_poisson_csc_workspace_bytes_f32(20000, 10, 96, 1) >= 8 * 20000 * 10
    p = _problem(G=20000, Fn=10, Ntot=96, E=1, seed=7, density=0.05)
    ll_r, g_r = _oracle(p)
    out, grads, _ = _run(p, SparseCounts.from_dense(p["y"]).to(DEV), dt)
    tol = 1e-11 if dt == torch.float64 else 3e-5
    assert relerr(out, ll_r) < tol
    for name, a, b in zip(("W", "V", "mean", "spread"), grads, g_r):
        assert relerr(a, b) < tol, (name, relerr(a, b))


@pytest.mark.parametrize("G", [300, 20000])
def test_csc_near_fit_precision(G):
    """y drawn from the model's own rate: sum t eps and u_f nearly cancel in d/dW; the fp32 gradient stays within 3e-5 of fp64."""
    from oracle import gpzoo_oracle as O
    N = 4000 if G == 300 else 200
    p = _problem(G=G, Fn=10, Ntot=N, E=1, seed=8, density=1.0)
    p["W"] = p["W"] - 3.0                                  # softplus(W) ~ 0.05-0.13: rates ~ 1, many zero counts
    nv = p["nvar"]
    sd = torch.cat((torch.clamp(p["spread"][:nv], min=5e-2).sqrt(), p["spread"][nv:]), 0)
    rate = O.poisson_rate(p["W"], p["mean"] + p["eps"] * sd, p["V"])[0]
    p["y"] = torch.poisson(rate, generator=torch.Generator().manual_seed(9))
    s = SparseCounts.from_dense(p["y"]).to(DEV)
    o64, g64, _ = _run(p, s, torch.float64)
    o32, g32, _ = _run(p, s, torch.float32)
    ll_r, g_r = _oracle(p)
    assert relerr(g64[0], g_r[0]) < 1e-10
    assert relerr(o32, o64) < 3e-5
    for name, a, b in zip(("W", "V", "mean", "spread"), g32, g64):
        assert relerr(a, b) < 3e-5, (name, relerr(a, b))


# ---- model level ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,dt", [("nsf_svgp_box", torch.float64), ("nsf_svgp_box", torch.float32),
                                     ("nsf_svgp_tc128", torch.float32)])
def test_nsf2_elbo_sparse_vs_reference_golden(name, dt):
    """NSF2.elbo with SparseCounts.from_dense(y) meets the golden tolerances of the dense test (1e-10 fp64, 1e-4 fp32)."""
    from tests.test_elbo_gpu import TOL, _check_grads, build_nsf
    inp, gout, ggrad = load_golden(name)
    model, named = build_nsf(inp, dt)
    y = SparseCounts.from_dense(inp["y"]).to(DEV)
    elbo, parts = model.elbo(inp["X"].to(DEV, dt), y, E=inp["eps"].shape[0], eps=inp["eps"].to(DEV, dt), return_parts=True)
    tol = TOL[dt]
    assert relerr(elbo, gout["elbo"]) < tol and relerr(parts["ll"], gout["ll"]) < tol
    (-elbo).backward()
    for p in named.values():
        p.grad.neg_()
    _check_grads(named, ggrad, tol)


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
def test_hybrid_nsf2_minibatch_sparse_vs_reference_golden(dt):
    import gpzoo_b200 as gz
    from tests.test_elbo_gpu import TOL, _P, _check_grads
    inp, gout, ggrad = load_golden("nsf_hybrid")
    L, M = inp["mu"].shape
    T = inp["Wcf"].shape[1]
    kern = gz.kernels.NSF_RBF(L=L)
    kern.sigma, kern.lengthscale = _P(inp["sigma"], dt), _P(inp["lengthscale"], dt)
    gp = gz.gp.SVGP(kern, dim=2, M=M, jitter=inp["jitter"])
    gp.Z, gp.mu, gp.Lu = _P(inp["Z"], dt), _P(inp["mu"], dt), _P(inp["Lu_raw"], dt)
    y = SparseCounts.from_dense(inp["y"]).to(DEV)
    prior = gz.gp.GaussianPrior(y, L=T)
    prior.mean, prior.scale = _P(inp["cf_mean"], dt), _P(inp["cf_scale"], dt)
    model = gz.likelihoods.Hybrid_NSF2(gp, prior, y, L=L, T=T)
    model.sf.W, model.cf.W, model.V = _P(inp["W"], dt), _P(inp["Wcf"], dt), _P(inp["V"], dt)
    idx = inp["idx"].to(DEV)
    eps = inp["eps"][:, :, inp["idx"]].to(DEV, dt)
    eps2 = inp["eps2"][:, :, inp["idx"]].to(DEV, dt)
    named = dict(Z=gp.Z, sigma=kern.sigma, lengthscale=kern.lengthscale, mu=gp.mu, Lu_raw=gp.Lu, W=model.sf.W,
                 V=model.V, Wcf=model.cf.W, cf_mean=prior.mean, cf_scale=prior.scale)
    elbo = model.elbo(inp["X"].to(DEV, dt), y, idx=idx, E=eps.shape[0], eps=eps, eps2=eps2)
    assert relerr(elbo, gout["elbo"]) < TOL[dt]
    (-elbo).backward()
    for p in named.values():
        p.grad.neg_()
    _check_grads(named, ggrad, TOL[dt])


@pytest.mark.parametrize("use_idx", [False, True])
def test_pnmf_elbo_sparse_matches_dense(use_idx):
    import gpzoo_b200 as gz
    dt = torch.float64
    p = _problem(G=40, Fn=3, Ntot=500, E=1, seed=10, density=0.2)
    y = p["y"].to(DEV, dt)
    ys = SparseCounts.from_dense(y)
    torch.manual_seed(0)
    prior = gz.gp.GaussianPrior(y, L=3)
    model = gz.likelihoods.PNMF(prior, y, L=3).to(DEV).double()
    idx = torch.randperm(500, generator=torch.Generator().manual_seed(1))[:300].to(DEV) if use_idx else None
    B = 500 if idx is None else 300
    eps = torch.randn(2, 3, B, generator=torch.Generator().manual_seed(2), dtype=dt).to(DEV)
    res = []
    for yy in (y, ys):
        model.zero_grad(set_to_none=True)
        e = model.elbo(yy, idx=idx, E=2, eps=eps)
        e.backward()
        res.append([e.detach()] + [q.grad.clone() for q in model.parameters() if q.grad is not None])
    assert len(res[0]) == len(res[1])
    for a, b in zip(res[1], res[0]):
        assert relerr(a, b) < 1e-10


def test_train_batched_sparse_matches_dense():
    """Five seeded utilities.train_batched steps: losses within 1e-5 relative of the dense-y run."""
    import gpzoo_b200 as gz
    from gpzoo_b200 import synthetic
    from tests.test_elbo_gpu import build_nsf
    prob = synthetic.nsf_problem(N=2048, M=64, L=4, G=64, E=1, seed=7, coord_scale=2.0, jitter=1e-2, dtype=torch.float32, device=DEV)
    model0, _ = build_nsf(prob, torch.float32)
    losses = []
    for y in (prob["y"], SparseCounts.from_dense(prob["y"])):
        model = copy.deepcopy(model0)
        opt = torch.optim.Adam(model.parameters(), lr=1e-2)
        torch.manual_seed(123)
        losses.append(gz.utilities.train_batched(model, opt, prob["X"], y, steps=5, E=2, batch_size=1000))
    assert len(losses[1]) == 5
    for a, b in zip(losses[1], losses[0]):
        assert abs(a - b) <= 1e-5 * abs(b), (losses[1], losses[0])
