"""The fused Gaussian factor-model ELBO (K7-G, gpz_gaussian_fwdbwd_* in csrc/gaussian.cu) and the RSF / FA models on the device.

The kernel is checked against float64 autograd of the closed-form expected log-likelihood (tests/test_gaussian_cpu.py, which also
pins that closed form to the Monte-Carlo mean of torch's Normal.log_prob).  Each output is checked as ||out - ref|| <= c ||mag||,
mag being the same sum over the absolute values of its summands, as in test_poisson_shapes_gpu.py: near a fit the residuals
cancel across spots, and sum_n t m against tau W V in d/dW."""
import math

import pytest
import torch
import torch.nn.functional as Fnn

from tests.test_gaussian_cpu import closed_form
from tests.test_poisson_shapes_gpu import SHAPES

DEV = "cuda"
OUTS = ("ll", "W", "bias", "noise", "mean", "spread")
# fp64: exact arithmetic throughout, partials summed in double.
C64 = 1e-10
# fp32: r = (y - b) - sum_f W m carries F + 2 roundings of |y| + |b| + sum |W m| (<= 2^-24 each), t = tau r one more; the
# contractions (F terms) and the per-CTA sums (32-gene chunks over a gene range of at most ~100 chunks, 64 spots per warp, four
# warps) are plain fp32 FMA, within (chunks + 64 + F) 2^-24 < 1e-5 of ||mag|| at these shapes; everything across CTAs, V, kappa,
# sum r^2 and the d/dW correction are double.  c = 1e-4 is the project's parity bar.
C32 = 1e-4
DTS = [torch.float32, torch.float64]


def _c(dt):
    return C64 if dt == torch.float64 else C32


def _raw(s):
    """noise with softplus(noise) = s, in float64."""
    s = torch.as_tensor(s, dtype=torch.float64)
    return s + torch.log(-torch.expm1(-s))


def _problem(G, Ntot, B, dt, F=10, nvar=None, seed=0, near=False):
    """Seeded inputs on the device, rounded to dt so the reference sees what the kernel sees.  Far from a fit: y ~ N(0, 4) against
    s ~ 0.3-3.  Near a fit: y drawn from the model at the factor means, mu = b + W m in about [0, 5], s_g from 0.05 to 1."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    rand = lambda *s: torch.rand(*s, generator=g, device=DEV, dtype=torch.float64)
    randn = lambda *s: torch.randn(*s, generator=g, device=DEV, dtype=torch.float64)
    idx = None if B is None else torch.randint(0, Ntot, (B,), generator=g, device=DEV)      # repeats included
    B = Ntot if B is None else B
    p = dict(idx=idx, W=randn(G, F), bias=randn(G), noise=randn(G), mean=0.3 * randn(F, B),
             spread=0.05 + 0.3 * rand(F, B), nvar=(F + 1) // 2 if nvar is None else nvar, cm=float(torch.tensor(5e-2, dtype=dt)))
    p["spread"][0, :7] = 1e-3                                  # below the variance clamp
    p["spread"][0, 7:9] = p["cm"]                              # at it: the gradient passes, as torch's clamp
    if near:
        assert idx is None
        p["W"] = 0.3 * randn(G, F)
        p["bias"] = 1.0 + 3.0 * rand(G)
        p["noise"] = _raw(torch.linspace(0.05, 1.0, G, dtype=torch.float64)).to(DEV)
    for k in ("W", "bias", "noise", "mean", "spread"):
        p[k] = p[k].to(dt).double()
    if near:
        s = Fnn.softplus(p["noise"])
        p["y"] = p["bias"][:, None] + p["W"] @ p["mean"] + s[:, None] * randn(G, Ntot)
    else:
        p["y"] = 2 * randn(G, Ntot)
    p["y"] = p["y"].to(dt).double()
    return p


def _kernel(p, y, dt):
    """GaussianLL on the device: ll and the gradients w.r.t. W, bias, noise, mean, spread."""
    from gpzoo_b200 import _cabi, functional as F
    lv = [p[k].to(dt).requires_grad_(True) for k in ("W", "bias", "noise", "mean", "spread")]
    _cabi.profile = {}
    try:
        out = F.GaussianLL.apply(y, p["idx"], *lv, p["nvar"], p["cm"])
    finally:
        calls, _cabi.profile = set(_cabi.profile), None
    assert "gaussian_fwdbwd" in calls, calls
    out.backward()
    return [out.detach()] + [t.grad for t in lv]


def _reference(p):
    """float64 autograd of the closed form, and each output's magnitude."""
    idx, nv, cm = p["idx"], p["nvar"], p["cm"]
    yb = p["y"] if idx is None else p["y"][:, idx]
    leaves = [p[k].clone().requires_grad_(True) for k in ("W", "bias", "noise", "mean", "spread")]
    ll = closed_form(yb, *leaves, nv, cm)
    ref = [ll.detach()] + list(torch.autograd.grad(ll, leaves))
    del ll
    with torch.no_grad():
        W, b, noise, m, spread = (p[k] for k in ("W", "bias", "noise", "mean", "spread"))
        B = m.shape[1]
        s = Fnn.softplus(noise)
        tau = 1 / s ** 2
        V = torch.cat((spread[:nv].clamp(min=cm), spread[nv:] ** 2), 0).sum(1)
        r = yb - b[:, None] - W @ m
        t = (tau[:, None] * r).abs()
        r2 = (r ** 2).sum(1)
        wv = (W ** 2 * V).sum(1)
        m_ll = (B * (0.5 * math.log(2 * math.pi) + s.log().abs()) + 0.5 * tau * (r2 + wv)).sum()
        m_W = t @ m.abs().t() + tau[:, None] * W.abs() * V
        m_b = t.sum(1)
        m_noise = torch.sigmoid(noise) * (B / s + (r2 + wv) / s ** 3)
        m_mean = W.abs().t() @ t
        kap = 0.5 * (W ** 2 * tau[:, None]).sum(0)
        m_spread = kap[:, None] * torch.cat((torch.ones_like(spread[:nv]), 2 * spread[nv:].abs()), 0)
    return ref, [m_ll, m_W, m_b, m_noise, m_mean, m_spread]


def _check(label, out, ref, mag, c):
    scaled = {k: (o.double() - r).norm().item() / max(m.norm().item(), 1e-300) for k, o, r, m in zip(OUTS, out, ref, mag)}
    worst = max(scaled, key=scaled.get)
    print(f"\n{label}: max ||out-ref||/||mag|| = {scaled[worst]:.2e} ({worst})")
    assert all(v <= c for v in scaled.values()), (label, scaled)


# ---- the call ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTS, ids=["f32", "f64"])
@pytest.mark.parametrize("case", list(SHAPES))
def test_shapes(case, dt):
    """Every shape of the Poisson shape table: gene-range splits, ragged chunks and ranges, a single range, odd B, idx with
    repeats (y_ld > B)."""
    s = SHAPES[case]
    p = _problem(s["G"], s["Ntot"], s["B"], dt, seed=21)
    out = _kernel(p, p["y"].to(dt), dt)
    ref, mag = _reference(p)
    _check(f"{case} {dt}", out, ref, mag, _c(dt))


FACTORS = (1, 10, 16, 17, 20, 32)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTS, ids=["f32", "f64"])
@pytest.mark.parametrize("F", FACTORS)
@pytest.mark.parametrize("nv", ["none", "all", "half"])
def test_factor_counts_and_nvar(F, nv, dt):
    nvar = dict(none=0, all=F, half=F // 2)[nv]
    s = SHAPES["idx_dup"]
    p = _problem(s["G"], s["Ntot"], s["B"], dt, F=F, nvar=nvar, seed=22)
    out = _kernel(p, p["y"].to(dt), dt)
    ref, mag = _reference(p)
    _check(f"F={F} n_var={nvar} {dt}", out, ref, mag, _c(dt))


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTS, ids=["f32", "f64"])
@pytest.mark.parametrize("case", ["cfg2", "odd_B"])
@pytest.mark.parametrize("F", [10, 20])
def test_near_fit(case, F, dt):
    """y drawn from the model (mu in about [0, 5], s_g from 0.05 to 1): the residuals are small against y."""
    s = SHAPES[case]
    p = _problem(s["G"], s["Ntot"], None, dt, F=F, seed=23, near=True)
    out = _kernel(p, p["y"].to(dt), dt)
    ref, mag = _reference(p)
    _check(f"near fit {case} F={F} {dt}", out, ref, mag, _c(dt))


@pytest.mark.gpu
def test_integer_y_and_column_slice():
    """Integer y is converted on the device; the C call reads a column slice of a wider matrix through y_ld > B without idx."""
    from gpzoo_b200._cabi import call, lib
    dt = torch.float32
    s = SHAPES["ragged_chunk"]
    p = _problem(s["G"], s["Ntot"], None, dt, seed=24)
    p["y"] = torch.randint(-50, 50, p["y"].shape, device=DEV, dtype=torch.int16).double()
    out = _kernel(p, p["y"].to(torch.int16), dt)
    ref, mag = _reference(p)
    _check("int16 y", out, ref, mag, C32)
    # columns [lo, hi) of the resident y: pointer offset by lo, y_ld = Ntot
    G, N = p["y"].shape
    lo, hi = 1000, 6001
    F = p["W"].shape[1]
    q = dict(p, mean=p["mean"][:, lo:hi].contiguous(), spread=p["spread"][:, lo:hi].contiguous())
    yf = p["y"].to(dt).contiguous()
    args = [q[k].to(dt).contiguous() for k in ("W", "bias", "noise", "mean", "spread")]
    ws_bytes = int(lib().gpz_gaussian_workspace_bytes_f32(G, F, hi - lo))
    ws = torch.empty(ws_bytes // 8 + 1, dtype=torch.float64, device=DEV)
    ll = torch.empty(1, dtype=torch.float64, device=DEV)
    outs = [torch.empty_like(args[0]), torch.empty_like(args[1]), torch.empty_like(args[2]), torch.empty_like(args[3]),
            torch.empty_like(args[4])]
    call("gaussian_fwdbwd", dt, yf.view(-1)[lo:], N, None, *args, G, F, hi - lo, q["nvar"], q["cm"], ll, *outs, ws, ws_bytes)
    q["y"] = p["y"][:, lo:hi]
    ref, mag = _reference(q)
    _check("column slice", [ll[0]] + outs, ref, mag, C32)


@pytest.mark.gpu
def test_empty_batch_and_unsupported():
    from gpzoo_b200 import _cabi, functional as F
    p = _problem(64, 300, None, torch.float64, seed=25)
    lv = [p[k].requires_grad_(True) for k in ("W", "bias", "noise")]
    out = F.GaussianLL.apply(p["y"], torch.zeros(0, dtype=torch.int64, device=DEV), *lv, p["mean"][:, :0], p["spread"][:, :0],
                             0, 0.0)
    out.backward()
    assert float(out) == 0.0 and all(float(t.grad.abs().sum()) == 0.0 for t in lv)
    W = torch.randn(64, 33, dtype=torch.float64, device=DEV)
    with pytest.raises(_cabi.GpzError, match="rc=-1001"):
        F.GaussianLL.apply(p["y"], None, W, p["bias"], p["noise"], torch.zeros(33, 300, dtype=torch.float64, device=DEV),
                           torch.ones(33, 300, dtype=torch.float64, device=DEV), 0, 0.0)


# ---- models --------------------------------------------------------------------------------------------------------------------
def _real_params(model, dt, seed):
    """Real loadings (both signs), intercepts and per-gene noise on the device."""
    g = torch.Generator().manual_seed(seed)
    G, L = model.W.shape
    model.W = torch.nn.Parameter(torch.randn(G, L, generator=g, dtype=torch.float64).to(DEV, dt))
    model.bias = torch.nn.Parameter((0.5 * torch.randn(G, generator=g, dtype=torch.float64)).to(DEV, dt))
    model.noise = torch.nn.Parameter(_raw(0.2 + torch.rand(G, generator=g, dtype=torch.float64)).to(DEV, dt))


def _model_y(model, mean, seed):
    """y drawn from the model at the factor means."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    with torch.no_grad():
        mu = model.bias.double()[:, None] + model.W.double() @ mean.double()
        s = Fnn.softplus(model.noise.double())[:, None]
        return mu + s * torch.randn(mu.shape, generator=g, device=DEV, dtype=torch.float64)


def _svgp_rsf(dt, N=1024, M=128, L=4, G=48, seed=3):
    import gpzoo_b200 as gz
    from gpzoo_b200 import synthetic
    prob = synthetic.nsf_problem(N=N, M=M, L=L, G=G, E=1, seed=seed, coord_scale=2.0, jitter=1e-2)
    dev = lambda t: t.to(DEV, dt)
    kern = gz.kernels.NSF_RBF(L=L)
    kern.sigma, kern.lengthscale = torch.nn.Parameter(dev(prob["sigma"])), torch.nn.Parameter(dev(prob["lengthscale"]))
    gp = gz.gp.SVGP(kern, dim=2, M=M, jitter=prob["jitter"])
    gp.Z, gp.mu, gp.Lu = (torch.nn.Parameter(dev(prob[k])) for k in ("Z", "mu", "Lu_raw"))
    model = gz.likelihoods.RSF(gp, prob["y"], L=L)
    _real_params(model, dt, seed)
    X = dev(prob["X"])
    with torch.no_grad():
        mean = gp.moments(X)["mean"]
    y = _model_y(model, mean, seed).to(dt)
    return model, X, y, prob


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTS, ids=["f32", "f64"])
def test_rsf_elbo_matches_oracle(dt):
    """RSF(SVGP) elbo (N = 1024, M = 128) equals the oracle's svgp moments + the float64 closed form - mvn_kl, value and every
    gradient (fp64 1e-10, fp32 1e-4)."""
    from oracle import gpzoo_oracle as O
    model, X, y, prob = _svgp_rsf(dt)
    _real_params(model, dt, 4)       # away from the fit: at it, d/dbias = sum_n t cancels to the fp32 rounding of the moments
    gp, kern = model.prior, model.prior.kernel
    named = dict(Z=gp.Z, sigma=kern.sigma, lengthscale=kern.lengthscale, mu=gp.mu, Lu_raw=gp.Lu, W=model.W, bias=model.bias,
                 noise=model.noise)
    elbo = model.elbo(X, y)
    grads = dict(zip(named, torch.autograd.grad(elbo, list(named.values()))))
    lv = {k: v.detach().double().clone().requires_grad_(True) for k, v in named.items()}
    Xd = X.double()
    Kzx = O.nsf_rbf(lv["Z"], Xd, lv["sigma"], lv["lengthscale"])
    Kzz = O.nsf_rbf(lv["Z"], lv["Z"], lv["sigma"], lv["lengthscale"])
    mean, var, Lu, Lc = O.svgp(O.rbf_diag(Xd, lv["sigma"]), Kzx, Kzz, lv["mu"], lv["Lu_raw"], gp.jitter, gp.clamp_min)
    ref = closed_form(y.double(), lv["W"], lv["bias"], lv["noise"], mean, var, mean.shape[0], gp.clamp_min) - O.mvn_kl(lv["mu"], Lu, Lc).sum()
    rgrads = dict(zip(lv, torch.autograd.grad(ref, list(lv.values()))))
    tol = _c(dt)
    rel = abs(float(elbo) - float(ref)) / abs(float(ref))
    gerr = {k: float((grads[k].double() - rgrads[k]).norm() / rgrads[k].norm()) for k in named}
    print(f"\nRSF vs oracle {dt}: elbo rel {rel:.1e}, gradients {gerr}")
    assert rel <= tol and max(gerr.values()) <= tol, (rel, gerr)


def _golden_prior(name, dt):
    """The prior of a golden NSF2 problem (VNNGP, MGGP_SVGP with groupsX, WSVGP) and its inputs."""
    import gpzoo_b200 as gz
    from tests.helpers import load_golden
    from tests.test_elbo_gpu import _P, _build_whitened, build_nsf
    inp, _, _ = load_golden(name)
    kw = {}
    if name == "nsf_vnngp":
        L, M = inp["mu"].shape
        kern = gz.kernels.NSF_RBF(L=L)
        kern.sigma, kern.lengthscale = _P(inp["sigma"], dt), _P(inp["lengthscale"], dt)
        gp = gz.gp.VNNGP(kern, dim=2, M=M, K=inp["K"], jitter=inp["jitter"])
        gp.Z, gp.mu, gp.Lu = _P(inp["Z"], dt), _P(inp["mu"], dt), _P(inp["Lu_raw"], dt)
    elif name == "nsf_wsvgp":
        _, gp, _ = _build_whitened(inp, dt)
    else:
        gp = build_nsf(inp, dt)[0].prior
        kw["groupsX"] = inp["groupsX"].to(DEV)
    return gp, inp["X"].to(DEV, dt), inp["y"], kw


@pytest.mark.gpu
@pytest.mark.parametrize("prior", ["nsf_vnngp", "nsf_mggp", "nsf_wsvgp", "fa"])
def test_elbo_ll_is_the_closed_form_of_forward_qF(prior):
    """RSF over VNNGP, MGGP_SVGP (groupsX) and WSVGP, and FA: elbo's ll equals the closed form evaluated from the qF forward()
    returns (fp64, 1e-10)."""
    import gpzoo_b200 as gz
    dt = torch.float64
    if prior == "fa":
        y0 = torch.randn(40, 700, dtype=dt)
        model = gz.likelihoods.FA(gz.gp.GaussianPrior(y0, L=5), y0, L=5).to(DEV, dt)
        _real_params(model, dt, 9)
        y = _model_y(model, model.prior.mean.detach(), 9)
        qF, pF = model.prior()
        ll = model.elbo(y) + torch.distributions.kl_divergence(qF, pF).sum()
        _, qF, _ = model(E=1)
    else:
        gp, X, y0, kw = _golden_prior(prior, dt)
        model = gz.likelihoods.RSF(gp, y0, L=gp.mu.shape[0])
        _real_params(model, dt, 8)
        with torch.no_grad():
            mean = model(X, E=1, **kw)[1].loc
        y = _model_y(model, mean, 8)
        ll = model.elbo(X, y, return_parts=True, **kw)[1]["ll"]
        _, qF, _, _ = model(X, E=1, **kw)
    ref = closed_form(y, model.W.double(), model.bias.double(), model.noise.double(), qF.loc.double(), qF.scale.double(), 0, 0.0)
    print(f"\n{prior}: ll {float(ll):.10e} closed form {float(ref):.10e}")
    assert abs(float(ll) - float(ref)) <= 1e-10 * abs(float(ref))


@pytest.mark.gpu
def test_forward_log_prob_converges_to_elbo_ll():
    """forward()'s pY.log_prob(y).mean(0).sum() over a large E agrees with elbo's ll within four standard errors."""
    dt = torch.float64
    torch.manual_seed(1)
    model, X, y, _ = _svgp_rsf(dt, N=512, M=64, L=3, G=20)
    ll = float(model.elbo(X, y, return_parts=True)[1]["ll"])
    per_draw = []
    with torch.no_grad():
        for _ in range(8):
            pY = model(X, E=500)[0]
            per_draw.append(pY.log_prob(y).sum((1, 2)))
    per_draw = torch.cat(per_draw)
    se = float(per_draw.std()) / math.sqrt(per_draw.numel())
    print(f"\nMC {float(per_draw.mean()):.6f} +- {se:.2e}, elbo ll {ll:.6f}")
    assert abs(float(per_draw.mean()) - ll) <= 4 * se


@pytest.mark.gpu
def test_two_spot_shards_sum_to_the_full_step():
    """Two spot shards with kl_weight = 0.5 sum to the full step's ELBO and shared gradients."""
    dt = torch.float64
    model, X, y, _ = _svgp_rsf(dt)
    N = X.shape[0]
    shared = [model.W, model.bias, model.noise, model.prior.mu, model.prior.Lu]
    full = model.elbo(X, y)
    gf = torch.autograd.grad(full, shared)
    parts, gs = 0.0, [torch.zeros_like(p) for p in shared]
    for lo, hi in ((0, N // 2), (N // 2, N)):
        e = model.elbo(X, y, idx=torch.arange(lo, hi, device=DEV), kl_weight=0.5)
        parts = parts + float(e)
        for acc, g in zip(gs, torch.autograd.grad(e, shared)):
            acc += g
    assert abs(parts - float(full)) <= 1e-10 * abs(float(full))
    for a, b in zip(gs, gf):
        assert float((a - b).norm() / b.norm()) <= 1e-10


@pytest.mark.gpu
def test_train_batched_keeps_negative_loadings():
    """train_batched on data generated with negative loadings lowers the loss and leaves negative entries in W (no clamp)."""
    import gpzoo_b200 as gz
    torch.manual_seed(0)
    model, X, y, _ = _svgp_rsf(torch.float32)
    _real_params(model, torch.float32, 99)                  # start away from the loadings, intercepts and noise y was drawn with
    assert bool((model.W < 0).any())
    opt = gz.optim.Adam(model.parameters(), lr=2e-2)
    losses = gz.utilities.train_batched(model, opt, X, y, steps=40, E=1, batch_size=512)
    for n, p in model.named_parameters():
        assert torch.isfinite(p).all(), n
    print(f"\nloss {losses[0]:.2f} -> {losses[-1]:.2f}")
    assert sum(losses[-5:]) < sum(losses[:5])
    assert bool((model.W < 0).any())
