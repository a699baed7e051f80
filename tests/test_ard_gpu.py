"""GPU: per-dimension (ARD) lengthscales for the four covariance kinds through the fused kernel build, its backward, the
split-FP16 plane writer and the models that take a stationary kernel.  The truth is float64 torch autograd of the
direct-difference ARD covariance below, with a square root that never sees 0 (the sub-gradient 0 at r = 0)."""
import math

import pytest
import torch

from tests.helpers import relerr

pytestmark = pytest.mark.gpu
DEV = "cuda"
KINDS = (0, 1, 2, 3)
NAMES = {0: "batched_ARD_RBF", 1: "batched_ARD_Matern32", 2: "batched_ARD_Matern12", 3: "batched_ARD_Matern52"}


def _tol(dt):
    return 1e-11 if dt == torch.float64 else 2e-5


def _q(t, step=2.0 ** -10):
    """Round to a multiple of `step`: coordinates and parameters that float32 holds exactly, so both precisions see one input."""
    return torch.round(t / step) * step


def _cov(x1, x2, sg, ls, kind):
    """K[l,i,j], float64, (L,) sigma and (L, D) lengthscales: the kind at unit lengthscale on s2 = sum_d (df_d / ls[l,d])^2."""
    df = x1[None, :, None, :] - x2[None, None, :, :]
    s2 = ((df / ls[:, None, None, :]) ** 2).sum(-1)
    pos = s2 > 0
    r = torch.where(pos, s2, torch.ones_like(s2)).sqrt() * pos
    sig2 = sg.reshape(-1, 1, 1) ** 2
    if kind == 0:
        return sig2 * torch.exp(-0.5 * s2)
    if kind == 2:
        return sig2 * torch.exp(-r)
    v = math.sqrt(3.0 if kind == 1 else 5.0) * r
    return sig2 * (1 + v + (v * v / 3 if kind == 3 else 0)) * torch.exp(-v)


def _kb(x1, x2, sg, ls, kind, jitter=0.0, want_lo=False):
    from gpzoo_b200 import functional as F
    return F.KernelBuild.apply(x1, x2, sg, ls, None, None, None, None, 1.0, jitter, want_lo, kind)


def _inputs(seed, n1, n2, D, L):
    """Lengthscales in [0.5, 2]: a factor of up to 4 between the axes of one factor."""
    g = torch.Generator().manual_seed(seed)
    x1 = _q(torch.randn(n1, D, generator=g, dtype=torch.float64))
    x2 = _q(torch.randn(n2, D, generator=g, dtype=torch.float64))
    sg = _q(1 + 0.1 * torch.rand(L, generator=g, dtype=torch.float64))
    ls = _q(0.5 + 1.5 * torch.rand(L, D, generator=g, dtype=torch.float64))
    return g, x1, x2, sg, ls


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("D", [1, 2, 3, 4])
@pytest.mark.parametrize("L", [1, 3, 33])
def test_forward_and_gradients(L, D, kind, dt):
    """n2 = 1030 is ragged against the 4-wide vectors; L = 33 takes several launches of the backward."""
    n1, n2 = 37, 1030
    g, x1, x2, sg, ls = _inputs(1000 * kind + 10 * D + L, n1, n2, D, L)
    Wt = torch.randn(L, n1, n2, generator=g, dtype=torch.float64)
    leaves = [t.clone().requires_grad_(True) for t in (x1, x2, sg, ls)]
    Kref = _cov(*leaves, kind)
    (Kref * Wt).sum().backward()
    dl = [t.to(DEV, dt).requires_grad_(True) for t in (x1, x2, sg, ls)]
    K = _kb(*dl, kind)
    assert K.shape == (L, n1, n2) and K.dtype == dt
    tol = _tol(dt)
    assert relerr(K, Kref) < tol
    (K * Wt.to(DEV, dt)).sum().backward()
    assert dl[3].grad.shape == (L, D)
    for name, r, c in zip(("x1", "x2", "sigma", "lengthscale"), leaves, dl):
        assert relerr(c.grad, r.grad) < tol, (name, relerr(c.grad, r.grad))


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("L", [3, 33])
def test_isotropic_limit(L, kind, dt):
    """ls[l, :] = ls_l: K and the x1 / x2 / sigma gradients are those of the isotropic call of the same kind, and the
    per-dimension lengthscale gradients sum to its lengthscale gradient."""
    n1, n2, D = 37, 1030, 3
    g, x1, x2, sg, ls = _inputs(300 + 10 * kind + L, n1, n2, D, L)
    ls1 = ls[:, 0].clone()
    Wt = torch.randn(L, n1, n2, generator=g, dtype=torch.float64).to(DEV, dt)
    iso = [t.to(DEV, dt).requires_grad_(True) for t in (x1, x2, sg, ls1)]
    ard = [t.to(DEV, dt).requires_grad_(True) for t in (x1, x2, sg, ls1[:, None].expand(L, D))]
    Ki, Ka = _kb(*iso, kind), _kb(*ard, kind)
    (Ki * Wt).sum().backward()
    (Ka * Wt).sum().backward()
    tol = _tol(dt)
    assert relerr(Ka, Ki) < tol
    for name, a, i in zip(("x1", "x2", "sigma"), ard, iso):
        assert relerr(a.grad, i.grad) < tol, name
    assert relerr(ard[3].grad.sum(1), iso[3].grad) < tol


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("kind", KINDS)
def test_kzz_coincident_and_near_coincident_points(kind, dt):
    """Kzz with jitter: the diagonal is exactly sigma^2 + jitter, and a diagonal-only upstream gradient gives exactly zero
    position and lengthscale gradients; pairs at r ~ 1e-4 of the smallest lengthscale, along single axes and diagonally,
    match the reference row by row."""
    L, n = 3, 37
    g, x, _, sg, ls = _inputs(50 + kind, n, 1, 3, L)
    near = 2.0 ** -14                                               # <= 1.2e-4 of the smallest lengthscale (0.5)
    x[1] = x[0] + torch.tensor([near, 0.0, 0.0], dtype=torch.float64)
    x[3] = x[2] + torch.tensor([0.0, 0.0, -near], dtype=torch.float64)
    x[5] = x[4] + torch.tensor([near, near, -near], dtype=torch.float64)
    jit = 0.05
    tol = _tol(dt)
    eye = torch.eye(n, dtype=torch.float64)
    for diag_only in (True, False):
        Wz = torch.randn(L, n, n, generator=g, dtype=torch.float64)
        if diag_only:
            Wz = Wz * eye
        leaves = [t.clone().requires_grad_(True) for t in (x, sg, ls)]
        Kref = _cov(leaves[0], leaves[0], leaves[1], leaves[2], kind) + jit * eye
        (Kref * Wz).sum().backward()
        zd, sd, ld = (t.to(DEV, dt).requires_grad_(True) for t in (x, sg, ls))
        K = _kb(zd, zd, sd, ld, kind, jitter=jit)
        assert relerr(K, Kref) < tol
        assert torch.equal(K.diagonal(dim1=-2, dim2=-1).cpu(), (sg.reshape(L, 1) ** 2 + jit).expand(L, n).to(dt))
        (K * Wz.to(DEV, dt)).sum().backward()
        assert bool(torch.isfinite(zd.grad).all()) and bool(torch.isfinite(ld.grad).all())
        if diag_only:
            assert int(torch.count_nonzero(zd.grad)) == 0
            assert int(torch.count_nonzero(ld.grad)) == 0
            assert relerr(sd.grad, leaves[1].grad) < tol
        else:
            assert relerr(zd.grad, leaves[0].grad) < tol
            for i in range(6):                                      # the near-coincident pairs alone
                assert relerr(zd.grad[i], leaves[0].grad[i]) < tol, i
            assert relerr(sd.grad, leaves[1].grad) < tol and relerr(ld.grad, leaves[2].grad) < tol


@pytest.mark.parametrize("kind", KINDS)
def test_tf32_lo_plane(kind):
    """want_lo: K - lo is exactly K truncated to tf32, and K is the same as without the lo plane."""
    _, x1, x2, sg, ls = _inputs(70 + kind, 37, 1030, 3, 3)
    args = [t.to(DEV, torch.float32) for t in (x1, x2, sg, ls)]
    K, lo = _kb(*args, kind, want_lo=True)
    trunc = (K.view(torch.int32) & -8192).view(torch.float32)        # 0xFFFFE000: sign, exponent, 10 mantissa bits
    assert torch.equal(K - lo, trunc)
    assert torch.equal(K, _kb(*args, kind))
    assert relerr(K, _cov(x1, x2, sg, ls, kind)) < 2e-5


@pytest.mark.parametrize("kind", KINDS)
def test_split_fp16_planes(kind):
    """KernelBuildH: (Kh + Kl) / sK within 2^-20 of sigma_l^2 of the float64 K, for a cross matrix and for Kzz with jitter."""
    from gpzoo_b200 import functional as F
    _, x1, x2, sg, ls = _inputs(80 + kind, 40, 1032, 2, 3)
    for a, b, jit in ((x1, x2, 0.0), (x1, x1, 0.05)):
        _, Kh, Kl, sK = F.KernelBuildH.apply(*(t.to(DEV, torch.float32) for t in (a, b, sg, ls)), None, None, None, None, 1.0, jit,
                                              kind, None)
        K = (Kh.float() + Kl.float()) / sK[:, None, None]
        ref = _cov(a, b, sg, ls, kind) + (jit * torch.eye(a.shape[0], dtype=torch.float64) if jit else 0.0)
        err = (K.double().cpu() - ref).abs().amax(dim=(1, 2)) / sg ** 2
        assert float(err.max()) <= 2.0 ** -20, err


def test_unsupported_arguments_are_rejected():
    """kind 4 and D = 5 return GPZ_ERR_UNSUPPORTED (-1001) from the ARD calls; groups with an L x D lengthscale are refused
    before the device."""
    from gpzoo_b200 import _cabi, functional as F
    from gpzoo_b200.kernels import embed_distance_matrix, _r2_table
    for dt in (torch.float32, torch.float64):
        _, x1, x2, sg, ls = _inputs(90, 16, 32, 2, 2)
        X, Z, s, l = (t.to(DEV, dt) for t in (x1, x2, sg, ls))
        with pytest.raises(_cabi.GpzError, match=r"rc=-1001"):
            _kb(X, Z, s, l, 4)
        if dt == torch.float32:
            with pytest.raises(_cabi.GpzError, match=r"rc=-1001"):
                F.KernelBuildH.apply(X, Z, s, l, None, None, None, None, 1.0, 0.0, 4, None)
        G = torch.ones(2, 16, 32, dtype=dt, device=DEV)
        with pytest.raises(_cabi.GpzError, match=r"rc=-1001"):
            F._kernel_build_bwd(X, Z, s, l, None, None, None, None, 1.0, 4, (True, True), G)
        _, x5, z5, _, l5 = _inputs(91, 16, 32, 5, 2)
        X5, Z5, L5 = (t.to(DEV, dt) for t in (x5, z5, l5))
        with pytest.raises(_cabi.GpzError, match=r"rc=-1001"):
            _kb(X5, Z5, s, L5, 0)
        with pytest.raises(_cabi.GpzError, match=r"rc=-1001"):
            F._kernel_build_bwd(X5, Z5, s, L5, None, None, None, None, 1.0, 0, (True, True), G)
        r2 = _r2_table(embed_distance_matrix(torch.ones(3, 3) - torch.eye(3)), dt).to(DEV)
        a = torch.ones(2, dtype=dt, device=DEV)
        gX, gZ = torch.arange(16, device=DEV) % 3, torch.arange(32, device=DEV) % 3
        with pytest.raises(_cabi.GpzError, match="multi-group"):
            F.KernelBuild.apply(X, Z, s, l, a, r2, gX, gZ, 1.0, 0.0, False, 0)


# ------------------------------------------------------------------------------------------------------------------------
# models
# ------------------------------------------------------------------------------------------------------------------------
def _P(t, dt):
    return torch.nn.Parameter(t.to(DEV, dt))


def _calls_of(fn):
    """Run fn() recording which C-ABI entry points it calls."""
    from gpzoo_b200 import _cabi
    _cabi.profile = {}
    try:
        out = fn()
    finally:
        prof, _cabi.profile = _cabi.profile, None
    return out, set(prof)


def _problem(kind, D, M):
    """Inducing points on a grid; lengthscales of one factor up to the grid spacing h and 4 times apart across the axes."""
    from gpzoo_b200 import synthetic
    prob = synthetic.nsf_problem(N=1024, M=M, L=3, G=32, D=D, E=1, seed=40 + 10 * D + kind, coord_scale=30.0, jitter=1e-1)
    h = 60.0 / round(M ** (1.0 / D))
    axes = torch.tensor([1.0, 0.25] if D == 2 else [1.0, 0.5, 0.25], dtype=torch.float64)
    prob["sigma"] = prob["sigma"].reshape(-1)
    prob["lengthscale"] = _q(h * torch.tensor([1.0, 0.9, 1.1], dtype=torch.float64)[:, None] * axes)
    return prob


def _model(prob, kind, dt, gp_cls="SVGP", lik="NSF2"):
    import gpzoo_b200 as gz
    D = prob["X"].shape[1]
    kern = getattr(gz.kernels, NAMES[kind])(dim=D)
    kern.sigma, kern.lengthscale = _P(prob["sigma"], dt), _P(prob["lengthscale"], dt)
    gp = getattr(gz.gp, gp_cls)(kern, dim=D, M=prob["Z"].shape[0], jitter=prob["jitter"])
    gp.Z, gp.mu, gp.Lu = _P(prob["Z"], dt), _P(prob["mu"], dt), _P(prob["Lu_raw"], dt)
    model = getattr(gz.likelihoods, lik)(gp, prob["y"], L=prob["mu"].shape[0])
    model.W, model.V = _P(prob["W"], dt), _P(prob["V"], dt)
    named = dict(Z=gp.Z, sigma=kern.sigma, lengthscale=kern.lengthscale, mu=gp.mu, Lu_raw=gp.Lu, W=model.W, V=model.V)
    if lik == "NSF2_NB":
        model.dispersion = _P(model.dispersion.detach(), dt)
        named["D"] = model.dispersion
    return model, named


def _step(model, named, prob, dt):
    elbo = model.elbo(prob["X"].to(DEV, dt), prob["y"].to(DEV, dt), E=1, eps=prob["eps"].to(DEV, dt))
    elbo.backward()
    return dict(elbo=elbo.detach(), **{k: v.grad.clone() for k, v in named.items()})


def _ref_step(prob, kind):
    """NSF2(SVGP(kernel)) restated in float64 torch: SVGP moments, Poisson log-likelihood with lgamma, KL(qU || pU)."""
    from oracle import gpzoo_oracle as O
    leaves = {k: prob[k].clone() for k in ("Z", "sigma", "lengthscale", "mu", "Lu_raw", "W", "V")}
    X, y, eps = prob["X"], prob["y"], prob["eps"]

    def terms():
        p = leaves
        Kzx = _cov(p["Z"], X, p["sigma"], p["lengthscale"], kind)
        Kzz = _cov(p["Z"], p["Z"], p["sigma"], p["lengthscale"], kind)
        Kxx = (p["sigma"] ** 2)[:, None].expand(-1, X.shape[0])
        mean, var, Lu, Lc = O.svgp(Kxx, Kzx, Kzz, p["mu"], p["Lu_raw"], prob["jitter"], 1e-6)
        rate = O.poisson_rate(p["W"], mean + eps * var.sqrt(), p["V"])
        ll = O.poisson_loglik(y, rate, True)
        return dict(elbo=ll - O.mvn_kl(p["mu"], Lu, Lc).sum())
    out, grads = O.value_and_grads(terms, leaves)
    return dict(elbo=out["elbo"], **grads)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("D", [2, 3])
@pytest.mark.parametrize("M", [128, 512])
def test_nsf2_svgp_fp32_vs_fp64_vs_restatement(M, D, kind):
    """NSF2(SVGP(ARD kernel)) at N = 1024, L = 3: the fp32 step runs the ARD split-FP16 plane writer and the tensor-core
    predictive op (M = 512 also the fp32 chain and the merged moments node, which launches the ARD backward early), within
    1e-4 of the fp64 step; the fp64 step is within 1e-10 of the float64 torch restatement."""
    prob = _problem(kind, D, M)
    res = {}
    for dt in (torch.float64, torch.float32):
        model, named = _model(prob, kind, dt)
        res[dt], calls = _calls_of(lambda: _step(model, named, prob, dt))
        if dt == torch.float32:
            want = {"kernel_build_ard_fwd_h", "svgp_predict_fwd_h", "svgp_predict_bwd_h"}
            if M > 256:
                want |= {"svgp_chain_bwd_s1"}
            assert want <= calls, calls
        assert "kernel_build_ard_bwd" in calls and "kernel_build_bwd" not in calls, calls
    errs = {k: relerr(res[torch.float32][k], res[torch.float64][k]) for k in res[torch.float64]}
    assert max(errs.values()) < 1e-4, errs
    ref = _ref_step(prob, kind)
    errs = {k: relerr(res[torch.float64][k], ref[k]) for k in ref}
    assert max(errs.values()) < 1e-10, errs


@pytest.mark.parametrize("kind", [0, 2])
def test_wsvgp_fp32_vs_fp64(kind):
    prob = _problem(kind, 2, 128)
    res = {}
    for dt in (torch.float64, torch.float32):
        model, named = _model(prob, kind, dt, gp_cls="WSVGP")
        res[dt] = _step(model, named, prob, dt)
    errs = {k: relerr(res[torch.float32][k], res[torch.float64][k]) for k in res[torch.float64]}
    assert max(errs.values()) < 1e-4, errs


@pytest.mark.parametrize("kind", [1, 3])
def test_nsf2_nb_fp32_vs_fp64(kind):
    prob = _problem(kind, 3, 128)
    res = {}
    for dt in (torch.float64, torch.float32):
        model, named = _model(prob, kind, dt, lik="NSF2_NB")
        res[dt] = _step(model, named, prob, dt)
    errs = {k: relerr(res[torch.float32][k], res[torch.float64][k]) for k in res[torch.float64]}
    assert max(errs.values()) < 1e-4, errs


@pytest.mark.parametrize("dt", [torch.float64, torch.float32])
@pytest.mark.parametrize("kind", [0, 3])
def test_predict_moments_matches_moments(kind, dt):
    prob = _problem(kind, 2, 128)
    model, _ = _model(prob, kind, dt)
    X = prob["X"].to(DEV, dt)
    with torch.no_grad():
        m = model.prior.moments(X)
    mean, var = model.prior.predict_moments(X, tile=384)
    tol = 1e-10 if dt == torch.float64 else 2e-5
    assert relerr(mean, m["mean"]) < tol and relerr(var, m["var"]) < tol


@pytest.mark.parametrize("kind", KINDS)
def test_project_to_inducing(kind):
    """initialisation.project_to_inducing: mu[l] = Kzz[l] (Kzx[l] Kxz[l] + j I)^-1 Kzx[l] f_l, float64."""
    import gpzoo_b200 as gz
    from gpzoo_b200 import initialisation as I
    g = torch.Generator().manual_seed(60 + kind)
    L, M, N, jit = 3, 36, 500, 1e-5
    ax = torch.linspace(-1, 1, 6, dtype=torch.float64)
    Z = torch.stack(torch.meshgrid(ax, ax, indexing="ij"), -1).reshape(M, 2)
    X = 2 * torch.rand(N, 2, generator=g, dtype=torch.float64) - 1
    f = torch.randn(L, N, generator=g, dtype=torch.float64)
    sg = torch.tensor([1.0, 1.2, 0.8], dtype=torch.float64)
    ls = torch.tensor([[0.4, 0.1], [0.6, 0.3], [0.9, 0.9]], dtype=torch.float64)
    kern = getattr(gz.kernels, NAMES[kind])(sigma=sg, lengthscale=ls).to(DEV).double()
    kern.sigma.data, kern.lengthscale.data = sg.to(DEV), ls.to(DEV)
    mu = I.project_to_inducing(kern, Z.to(DEV), X.to(DEV), f.to(DEV), jitter=jit)
    Kzx, Kzz = _cov(Z, X, sg, ls, kind), _cov(Z, Z, sg, ls, kind)
    A = Kzx @ Kzx.transpose(-1, -2) + jit * torch.eye(M, dtype=torch.float64)
    ref = (Kzz @ torch.linalg.solve(A, Kzx @ f[:, :, None]))[:, :, 0]
    assert mu.shape == (L, M)
    assert relerr(mu, ref) < 1e-6
