"""The fused negative-binomial ELBO (K7-NB, gpz_negbin_fwdbwd_* in csrc/poisson.cu) against a float64 autograd reference on the
device: torch.distributions.NegativeBinomial(total_count=theta, logits=log r - log theta).log_prob(y) over oracle.poisson_rate.

Each output is checked as ||out - ref|| <= c ||mag||, mag being the same sum over the absolute values of the summands of the
stable form (|theta log1p(r / theta)|, never theta log theta), as in test_poisson_shapes_gpu.py."""
import math
import time

import pytest
import torch
import torch.nn.functional as Fnn

from tests.test_poisson_shapes_gpu import SHAPES, _problem, _sd

DEV = "cuda"
OUTS = ("ll", "W", "V", "mean", "spread", "D")
THETAS = (0.05, 1.0, 50.0, 1e4, 1e6)

# fp64: exact log, log1p, lgamma and division; the tables are sums of at most 63 exact logs / reciprocals in double.
C64 = 1e-10
# fp32, tensor-core path (F <= 16): as for Poisson, the split-bf16 products carry 1.1e-5 each and two contractions 2.3e-5 of
# ||mag|| to first order.  The element step adds __log2f (2^-22 absolute near 1, so <= 5e-6 relative on log1p above the series'
# threshold of 1/32; the series itself is exact to 5e-9), rcp.approx (1 ulp) and the tables rounded from double to fp32 (6e-8
# relative of |Lambda|, |Psi|, each a term of mag).  The fp32 sums (at most ~1200 CTA partials, 8 warps, 64-gene chunks) grow as
# sqrt(n) 2^-24 < 3e-6.  poisson_kernel2 (F > 16) is plain fp32 FMA with __logf / __fdividef: within 1.5e-5.  Total < 3.5e-5;
# c = 1e-4 leaves the margin the project's parity bar allows and is still far below what a dropped block or gene range moves.
C32 = 1e-4


@pytest.fixture(scope="module", autouse=True)
def _report():
    t0 = time.perf_counter()
    if torch.cuda.is_available():
        torch.cuda.reset_peak_memory_stats()
    yield
    if torch.cuda.is_available():
        print(f"\n[negbin] {time.perf_counter() - t0:.1f} s, peak max_memory_allocated "
              f"{torch.cuda.max_memory_allocated() / 2**30:.2f} GiB")


def _raw_dispersion(theta):
    """D with softplus(D) = theta, in float64."""
    theta = torch.as_tensor(theta, dtype=torch.float64)
    return torch.where(theta > 20, theta, theta + torch.log(-torch.expm1(-theta)))


def _with_theta(p, dt, thetas=THETAS):
    """Per-gene dispersion cycling through `thetas` (rounded to dt)."""
    G = p["W"].shape[0]
    th = torch.tensor(thetas, dtype=torch.float64, device=DEV)[torch.arange(G, device=DEV) % len(thetas)]
    p["D"] = _raw_dispersion(th).to(dt).double()
    return p


def _kernel(p, y, dt, with_lgamma=True, entry="negbin_fwdbwd"):
    from gpzoo_b200 import _cabi, functional as F
    lv = [p[k].to(dt).requires_grad_(True) for k in ("W", "V", "mean", "spread", "D")]
    W, V, mean, spread, D = lv
    _cabi.profile = {}
    try:
        out = F.NegBinLL.apply(y, p["idx"], W, V, D, mean, spread, p["eps"].to(dt), p["nvar"], p["cm"], p["soft"], with_lgamma)
    finally:
        calls, _cabi.profile = set(_cabi.profile), None
    assert entry in calls, calls
    out.backward()
    return [out.detach()] + [W.grad, V.grad, mean.grad, spread.grad, D.grad]


def nb_log_prob(y, rate, theta, with_lgamma=True):
    """torch's NegativeBinomial.log_prob with total_count = theta, logits = log r - log theta (mean r)."""
    lp = distributions_nb(theta, rate).log_prob(y)
    if not with_lgamma:
        lp = lp + torch.lgamma(y + 1)
    return lp


def distributions_nb(theta, rate):
    return torch.distributions.NegativeBinomial(total_count=theta, logits=rate.log() - theta.log(), validate_args=False)


def _log_prob64(pY, y):
    """pY.log_prob(y) of a forward() NegativeBinomial, evaluated in float64 (differentiably): in fp32, torch's
    lgamma(y + theta) - lgamma(theta) loses about 1 per element at theta = 1e6."""
    nb = torch.distributions.NegativeBinomial(total_count=pY.total_count.double(), logits=pY.logits.double(), validate_args=False)
    return nb.log_prob(y.double())


def _reference(p, with_lgamma=True, y=None):
    from oracle import gpzoo_oracle as O
    y = p["y"] if y is None else y
    idx, eps, soft, E, nv = p["idx"], p["eps"], p["soft"], p["E"], p["nvar"]
    leaves = [p[k].clone().requires_grad_(True) for k in ("W", "V", "mean", "spread", "D")]
    Wl, Vl, ml, sl, Dl = leaves
    rate = O.poisson_rate(Wl, ml + eps * _sd(p, sl), Vl if idx is None else Vl[idx], softplus_W=soft)
    yb = (y if idx is None else y[:, idx]).double()
    theta = Fnn.softplus(Dl)[:, None]
    ll = nb_log_prob(yb, rate, theta, with_lgamma).mean(0).sum()
    ref = [ll.detach()] + list(torch.autograd.grad(ll, leaves))
    del ll
    with torch.no_grad():
        r = rate.detach()
        del rate
        th = theta.detach()
        W, V, spread, D = p["W"], p["V"], p["spread"], p["D"]
        Vb = V if idx is None else V[idx]
        spV = Fnn.softplus(Vb)
        sd = _sd(p, spread)
        ef = spV * torch.exp(p["mean"] + eps * sd)
        w = (Fnn.softplus(W) if soft else W).abs()
        dw = torch.sigmoid(W) if soft else torch.ones_like(W)
        l1p = torch.log1p(r / th)
        m_ll = ((torch.lgamma(yb + th) - torch.lgamma(th)).abs() + torch.xlogy(yb, r / (th + r)).abs() + th * l1p).sum() / E
        if with_lgamma:
            m_ll = m_ll + torch.lgamma(yb + 1).sum()
        a = th * (yb + r) / (r * (th + r)) / E                          # >= |d ll / d r|
        m_W = torch.matmul(a, ef.transpose(1, 2)).sum(0) * dw
        u = torch.matmul(w.t(), a)
        m_mean = (ef * u).sum(0)
        m_spread = (ef * eps.abs() * u).sum(0)
        m_spread[:nv] *= torch.where(spread[:nv] >= p["cm"], 1 / (2 * sd[:nv]), torch.zeros_like(sd[:nv]))
        m_Vb = torch.sigmoid(Vb) / spV * (a * r).sum((0, 1))
        m_V = m_Vb if idx is None else torch.zeros_like(V).index_add_(0, idx, m_Vb)
        m_D = torch.sigmoid(D) * ((torch.digamma(yb + th) - torch.digamma(th)).abs() + l1p + (r - yb).abs() / (th + r)).sum((0, 2)) / E
    return ref, [m_ll, m_W, m_V, m_mean, m_spread, m_D]


def _check(label, out, ref, mag, c):
    scaled = {k: (o.double() - r).norm().item() / m.norm().item() for k, o, r, m in zip(OUTS, out, ref, mag)}
    worst = max(scaled, key=scaled.get)
    print(f"\n{label}: max ||out-ref||/||mag|| = {scaled[worst]:.2e} ({worst})")
    assert all(v <= c for v in scaled.values()), (label, scaled)


def _c(dt):
    return C64 if dt == torch.float64 else C32


DTS = [torch.float32, torch.float64]


def _nb_counts(p, g):
    """Counts drawn from NB(r, theta) at the reference's first-sample rate (a gamma-Poisson mixture): data near a fit."""
    from oracle import gpzoo_oracle as O
    rate = O.poisson_rate(p["W"], p["mean"] + p["eps"] * _sd(p, p["spread"]), p["V"], softplus_W=p["soft"]).mean(0)
    th = Fnn.softplus(p["D"])[:, None]
    lam = torch._standard_gamma(th.expand_as(rate).contiguous(), generator=g) * rate / th
    return torch.poisson(lam, generator=g)


# ---- grid shapes ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTS, ids=["f32", "f64"])
@pytest.mark.parametrize("case", ["cfg2", "ragged_chunk", "single_range", "cfg4_idx", "idx_dup"])
def test_gene_range_splits(case, dt):
    s = SHAPES[case]
    p = _with_theta(_problem(s["G"], s["Ntot"], s["B"], s["E"], dt, seed=11), dt)
    out = _kernel(p, p["y"].to(dt), dt)
    ref, mag = _reference(p)
    _check(f"{case} {dt}", out, ref, mag, _c(dt))


@pytest.mark.gpu
@pytest.mark.parametrize("dt,F", [(torch.float32, f) for f in (1, 10, 16, 17, 20, 32)] + [(torch.float64, f) for f in (1, 5, 13, 21, 32)],
                         ids=[f"f32-F{f}" for f in (1, 10, 16, 17, 20, 32)] + [f"f64-F{f}" for f in (1, 5, 13, 21, 32)])
def test_factor_counts(dt, F):
    s = SHAPES["ragged_chunk"]
    p = _with_theta(_problem(s["G"], s["Ntot"], s["B"], s["E"], dt, F=F, seed=12), dt)
    out = _kernel(p, p["y"].to(dt), dt)
    ref, mag = _reference(p)
    _check(f"F={F} {dt}", out, ref, mag, _c(dt))


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTS, ids=["f32", "f64"])
@pytest.mark.parametrize("theta", THETAS)
def test_single_dispersion(theta, dt):
    s = SHAPES["ragged_chunk"]
    p = _with_theta(_problem(s["G"], s["Ntot"], s["B"], s["E"], dt, seed=13), dt, (theta,))
    out = _kernel(p, p["y"].to(dt), dt)
    ref, mag = _reference(p)
    _check(f"theta={theta} {dt}", out, ref, mag, _c(dt))


# ---- counts --------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["float", "uint8", "int16", "int32", "float_nonint", "no_lgamma", "near_fit"])
def test_counts_cfg2_fp32(kind):
    s = SHAPES["cfg2"]
    dt = torch.float32
    p = _with_theta(_problem(s["G"], s["Ntot"], s["B"], s["E"], dt, seed=14, near=kind == "near_fit"), dt)
    g = torch.Generator(device=DEV).manual_seed(15)
    y = p["y"]
    entry = "negbin_fwdbwd"
    if kind in ("float", "uint8", "int16", "int32"):
        top = 256 if kind == "uint8" else 4000                      # counts >= 64 take nb_slow
        big = torch.rand(y.shape, generator=g, device=DEV) < 0.01
        y = p["y"] = torch.where(big, torch.randint(64, top, y.shape, generator=g, device=DEV, dtype=torch.float64), y)
        if kind != "float":
            y = y.to(getattr(torch, kind))
            entry = "negbin_fwdbwd_yt"
    elif kind == "float_nonint":
        y = p["y"] = 3 * torch.rand(y.shape, generator=g, device=DEV, dtype=torch.float64).to(dt).double()
    elif kind == "near_fit":
        y = p["y"] = _nb_counts(p, g)
    with_lgamma = kind != "no_lgamma"
    out = _kernel(p, y.to(dt) if y.is_floating_point() else y, dt, with_lgamma=with_lgamma, entry=entry)
    ref, mag = _reference(p, with_lgamma=with_lgamma)
    _check(f"cfg2 {kind}", out, ref, mag, C32)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["big_and_nonint", "near_fit", "no_lgamma"])
def test_counts_fp64(kind):
    s = SHAPES["ragged_chunk"]
    dt = torch.float64
    p = _with_theta(_problem(s["G"], s["Ntot"], s["B"], s["E"], dt, seed=16), dt)
    g = torch.Generator(device=DEV).manual_seed(17)
    if kind == "big_and_nonint":
        y = p["y"]
        big = torch.rand(y.shape, generator=g, device=DEV) < 0.01
        y = torch.where(big, torch.randint(64, 4000, y.shape, generator=g, device=DEV, dtype=torch.float64), y)
        frac = torch.rand(y.shape, generator=g, device=DEV) < 0.01
        p["y"] = torch.where(frac, 5 * torch.rand(y.shape, generator=g, device=DEV, dtype=torch.float64), y)
    elif kind == "near_fit":
        p["y"] = _nb_counts(p, g)
    with_lgamma = kind != "no_lgamma"
    out = _kernel(p, p["y"], dt, with_lgamma=with_lgamma)
    ref, mag = _reference(p, with_lgamma=with_lgamma)
    _check(f"fp64 {kind}", out, ref, mag, C64)


# ---- the Poisson limit ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_poisson_limit_fp64():
    """theta = 1e8: ll and the W, V, mean, spread gradients agree with the dense Poisson call to 1e-6 relative."""
    from gpzoo_b200 import functional as F
    from tests.helpers import relerr
    s = SHAPES["ragged_chunk"]
    dt = torch.float64
    p = _with_theta(_problem(s["G"], s["Ntot"], s["B"], s["E"], dt, seed=18), dt, (1e8,))
    nb = _kernel(p, p["y"], dt)
    lv = [p[k].detach().clone().requires_grad_(True) for k in ("W", "V", "mean", "spread")]
    po = F.PoissonLL.apply(p["y"], p["idx"], *lv, p["eps"], p["nvar"], p["cm"], p["soft"], True)
    po.backward()
    for name, a, b in zip(OUTS[:5], nb[:5], [po.detach()] + [t.grad for t in lv]):
        assert relerr(a, b) < 1e-6, (name, relerr(a, b))


# ---- digamma / lgamma ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fn", ["digamma", "lgamma"])
def test_digamma_lgamma_match_torch(fn):
    from gpzoo_b200._cabi import call
    x = torch.logspace(-3, 4, 3001, dtype=torch.float64, device=DEV)
    out = torch.empty_like(x)
    call(fn, torch.float64, x, out, x.numel())
    ref = getattr(torch, fn)(x)
    # lgamma has roots at x = 1 and 2, where its error is bounded in absolute terms
    scale = ref.abs() if fn == "digamma" else ref.abs().clamp(min=1.0)
    err = ((out - ref).abs() / scale).max().item()
    print(f"\n{fn}: max error {err:.2e}")
    assert err <= 1e-13


# ---- models --------------------------------------------------------------------------------------------------------------------
def _svgp_model(dt, N=1024, M=128, L=4, G=48, seed=3):
    import gpzoo_b200 as gz
    from gpzoo_b200 import synthetic
    prob = synthetic.nsf_problem(N=N, M=M, L=L, G=G, E=1, seed=seed, coord_scale=2.0, jitter=1e-2)
    dev = lambda t: t.to(DEV, dt)
    kern = gz.kernels.NSF_RBF(L=L)
    kern.sigma, kern.lengthscale = torch.nn.Parameter(dev(prob["sigma"])), torch.nn.Parameter(dev(prob["lengthscale"]))
    gp = gz.gp.SVGP(kern, dim=2, M=M, jitter=prob["jitter"])
    gp.Z, gp.mu, gp.Lu = (torch.nn.Parameter(dev(prob[k])) for k in ("Z", "mu", "Lu_raw"))
    model = gz.likelihoods.NSF2_NB(gp, prob["y"], L=L)
    model.W, model.V = torch.nn.Parameter(dev(prob["W"])), torch.nn.Parameter(dev(prob["V"]))
    g = torch.Generator().manual_seed(seed)
    model.dispersion = torch.nn.Parameter(dev(_raw_dispersion(torch.tensor(THETAS, dtype=torch.float64)[torch.arange(G) % 5])
                                              + 0.1 * torch.randn(G, generator=g, dtype=torch.float64)))
    return model, dev(prob["X"]), dev(prob["y"])


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTS, ids=["f32", "f64"])
def test_nsf2_nb_elbo_matches_forward(dt):
    """NSF2_NB.elbo equals pY.log_prob(y).mean(0).sum() - KL from forward() with the same eps (log_prob taken in float64); the
    gradients too."""
    model, X, y = _svgp_model(dt)
    L, N = model.W.shape[1], X.shape[0]
    eps = torch.randn(2, L, N, dtype=dt, device=DEV, generator=torch.Generator(device=DEV).manual_seed(5))
    params = [p for p in model.parameters() if p.requires_grad]
    elbo = model.elbo(X, y, E=2, eps=eps)
    g1 = torch.autograd.grad(elbo, params, allow_unused=True)
    pY, qF, qU, pU = model(X, E=2, eps=eps)
    ref = _log_prob64(pY, y).mean(0).sum() - torch.distributions.kl_divergence(qU, pU).sum()
    g2 = torch.autograd.grad(ref, params, allow_unused=True)
    tol = 1e-10 if dt == torch.float64 else 1e-4
    assert abs(float(elbo) - float(ref)) <= tol * abs(float(ref)), (float(elbo), float(ref))
    for a, b in zip(g1, g2):
        if a is None and b is None:
            continue
        err = float((a.double() - b.double()).norm() / b.double().norm().clamp(min=1e-30))
        assert err <= tol, err
    assert g1[[i for i, p in enumerate(params) if p is model.dispersion][0]].abs().sum() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTS, ids=["f32", "f64"])
def test_nsf2_nb_elbo_matches_oracle(dt):
    """NSF2_NB.elbo over SVGP (N = 1024, M = 128: the fp32 step runs the tensor-core kernels) equals the oracle's svgp moments +
    the float64 NB reference - mvn_kl, value and every gradient, dD included (fp64 1e-10, fp32 1e-4)."""
    from oracle import gpzoo_oracle as O
    model, X, y = _svgp_model(dt)
    L, N = model.W.shape[1], X.shape[0]
    eps = torch.randn(2, L, N, dtype=torch.float64, device=DEV, generator=torch.Generator(device=DEV).manual_seed(8)).to(dt)
    gp, kern = model.prior, model.prior.kernel
    named = dict(Z=gp.Z, sigma=kern.sigma, lengthscale=kern.lengthscale, mu=gp.mu, Lu_raw=gp.Lu, W=model.W, V=model.V,
                 D=model.dispersion)
    elbo = model.elbo(X, y, E=2, eps=eps)
    grads = dict(zip(named, torch.autograd.grad(elbo, list(named.values()))))
    leaves = {k: v.detach().double().clone().requires_grad_(True) for k, v in named.items()}
    p = O.NSFParams(**{k: leaves[k] for k in ("Z", "sigma", "lengthscale", "mu", "Lu_raw", "W", "V")}, jitter=gp.jitter)
    terms = O.nsf_svgp_terms(p, X.double(), y.double(), eps.double())
    theta = Fnn.softplus(leaves["D"])[:, None]
    ref = nb_log_prob(y.double(), terms["rate"], theta).mean(0).sum() - terms["kl"].sum()
    rgrads = dict(zip(leaves, torch.autograd.grad(ref, list(leaves.values()))))
    tol = 1e-10 if dt == torch.float64 else 1e-4
    rel = abs(float(elbo) - float(ref)) / abs(float(ref))
    gerr = {k: float((grads[k].double() - rgrads[k]).norm() / rgrads[k].norm()) for k in named}
    print(f"\nNSF2_NB vs oracle {dt}: elbo rel {rel:.1e}, gradients {gerr}")
    assert rel <= tol and max(gerr.values()) <= tol, (rel, gerr)


@pytest.mark.gpu
def test_pnmf_nb_and_hybrid_nb_f20():
    """PNMF_NB and Hybrid_NSF2_NB (L + T = 20 factors: the fp32 CUDA-core path) against forward()'s NegativeBinomial."""
    import gpzoo_b200 as gz
    dt = torch.float32
    model, X, y = _svgp_model(dt, L=10, G=40)
    N = X.shape[0]
    gen = torch.Generator(device=DEV).manual_seed(6)
    prior = gz.gp.GaussianPrior(y, L=10).to(DEV)
    hyb = gz.likelihoods.Hybrid_NSF2_NB(model.prior, prior, y, L=10, T=10).to(DEV)
    hyb.dispersion.data = model.dispersion.data.clone()
    eps, eps2 = (torch.randn(1, 10, N, dtype=dt, device=DEV, generator=gen) for _ in range(2))
    e1 = hyb.elbo(X, y, E=1, eps=eps, eps2=eps2)
    pY, qF1, qU, pU, qF2, pF2 = hyb(X, E=1, eps=eps, eps2=eps2)
    r1 = (_log_prob64(pY, y).mean(0).sum() - torch.distributions.kl_divergence(qU, pU).sum()
          - torch.distributions.kl_divergence(qF2, pF2).sum())
    assert abs(float(e1) - float(r1)) <= 1e-4 * abs(float(r1)), (float(e1), float(r1))
    pn = gz.likelihoods.PNMF_NB(gz.gp.GaussianPrior(y, L=5).to(DEV), y, L=5).to(DEV)
    eps = torch.randn(2, 5, N, dtype=dt, device=DEV, generator=gen)
    e2 = pn.elbo(y, E=2, eps=eps)
    pY, qF, pF = pn(E=2, eps=eps)
    r2 = _log_prob64(pY, y).mean(0).sum() - torch.distributions.kl_divergence(qF, pF).sum()
    assert abs(float(e2) - float(r2)) <= 1e-4 * abs(float(r2)), (float(e2), float(r2))


@pytest.mark.gpu
def test_two_spot_shards_sum_to_the_full_step():
    """Two spot shards with kl_weight = 0.5 sum to the full step's ELBO and shared gradients (dD included)."""
    dt = torch.float64
    model, X, y = _svgp_model(dt)
    L, N = model.W.shape[1], X.shape[0]
    eps = torch.randn(1, L, N, dtype=dt, device=DEV, generator=torch.Generator(device=DEV).manual_seed(7))
    shared = [model.W, model.dispersion, model.prior.mu, model.prior.Lu]
    full = model.elbo(X, y, E=1, eps=eps)
    gf = torch.autograd.grad(full, shared)
    parts, gs = 0.0, [torch.zeros_like(p) for p in shared]
    for lo, hi in ((0, N // 2), (N // 2, N)):
        idx = torch.arange(lo, hi, device=DEV)
        e = model.elbo(X, y, idx=idx, E=1, eps=eps[:, :, lo:hi], kl_weight=0.5)
        parts = parts + float(e)
        for acc, g in zip(gs, torch.autograd.grad(e, shared)):
            acc += g
    assert abs(parts - float(full)) <= 1e-10 * abs(float(full))
    for a, b in zip(gs, gf):
        assert float((a - b).norm() / b.norm()) <= 1e-10


@pytest.mark.gpu
def test_train_batched_moves_dispersion():
    import gpzoo_b200 as gz
    model, X, y = _svgp_model(torch.float32)
    d0 = model.dispersion.detach().clone()
    opt = gz.optim.Adam(model.parameters(), lr=1e-2, clamp_nonneg=[model.W])
    gz.utilities.train_batched(model, opt, X, y, steps=5, E=1, batch_size=512)
    for n, p in model.named_parameters():
        assert torch.isfinite(p).all(), n
    assert not torch.equal(model.dispersion.detach(), d0)
