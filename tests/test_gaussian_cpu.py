"""CPU: the Gaussian factor-model likelihood's C ABI (gpz_gaussian_*), the workspace size the library reports, the RSF / FA model
classes' parameters and input checks, and the closed-form expected log-likelihood the GPU tests compare against."""
import math
import os

import pytest
import torch
import torch.nn.functional as Fnn

from gpzoo_b200.counts import SparseCounts

from tests.test_poisson_shapes_gpu import SHAPES, poisson_grid

NEW_SYMBOLS = ("gpz_gaussian_workspace_bytes_f32", "gpz_gaussian_workspace_bytes_f64", "gpz_gaussian_fwdbwd_f32",
               "gpz_gaussian_fwdbwd_f64")


def _lib():
    from gpzoo_b200 import _cabi, build
    if not os.path.exists(_cabi.LIB_PATH):
        build.build()
    return _cabi.lib()


def closed_form(y, W, bias, noise, mean, spread, n_var, clamp_min):
    """sum_{g,n} E_q[log N(y_gn | bias_g + sum_f W_gf F_fn, softplus(noise_g)^2)] under q(F) = N(mean, v), in closed form:
    v = clamp(spread, clamp_min) for f < n_var, spread^2 otherwise.  Differentiable torch ops, in the inputs' dtype."""
    s = Fnn.softplus(noise)
    v = torch.cat((spread[:n_var].clamp(min=clamp_min), spread[n_var:] ** 2), 0)
    r = y - bias[:, None] - W @ mean
    ll = (-0.5 * math.log(2 * math.pi) - torch.log(s)[:, None] - 0.5 * r ** 2 / (s ** 2)[:, None]).sum()
    return ll - 0.5 * ((W ** 2 / (s ** 2)[:, None]) * v.sum(1)[None, :]).sum()


def _gaussian_workspace_bytes(G, F, B, is_f32):
    """Mirror of gauss_ws_bytes in csrc/gaussian.cu: V and kappa [2][F] (double) | the genes' ll [G] (double) | sum t, sum t^2
    partials [nbx][G][2] (double) | d/dW partials [nbx][G][F] | d/dmean partials [nby][F][B], each 16-byte aligned.  The grid
    is poisson_kernel2's (the "k2" path of the mirror)."""
    _, nbx, nby, _ = poisson_grid(G, F, B, False)
    elt = 4 if is_f32 else 8
    a16 = lambda n: -(-n // 16) * 16
    return a16(16 * F) + a16(8 * G) + 16 * nbx * G + a16(elt * nbx * G * F) + a16(elt * nby * F * B)


def test_header_exports_and_abi_version():
    from gpzoo_b200 import _cabi
    lib = _lib()
    assert lib.gpz_abi_version() == 4                      # entry points were only added
    syms = _cabi.exported_symbols()
    for s in NEW_SYMBOLS:
        assert s in syms, s
        assert hasattr(lib, s), s


def test_gaussian_workspace_bytes_match_the_mirror():
    lib = _lib()
    for s in SHAPES.values():
        for F in (1, 10, 16, 17, 20, 32):
            for is_f32, suf in ((True, "f32"), (False, "f64")):
                args = (s["G"], F, s["B"] or s["Ntot"])
                got = getattr(lib, "gpz_gaussian_workspace_bytes_" + suf)(*args)
                assert got == _gaussian_workspace_bytes(*args, is_f32), (args, suf)


def _models(y):
    import gpzoo_b200 as gz
    kern = gz.kernels.NSF_RBF(L=3)
    gp = gz.gp.SVGP(kern, dim=2, M=8)
    prior = gz.gp.GaussianPrior(y, L=2)
    return ((gz.likelihoods.RSF, gp, dict(L=3)), (gz.likelihoods.FA, prior, dict(L=2)))


def test_state_dict_is_the_prior_plus_w_bias_noise():
    y = torch.randn(7, 30)
    for cls, prior, kw in _models(y):
        m = cls(prior, y, **kw)
        keys = set(m.state_dict())
        assert keys == {"prior." + k for k in prior.state_dict()} | {"W", "bias", "noise"}, (cls.__name__, keys)
        assert tuple(m.W.shape) == (7, kw["L"]) and tuple(m.bias.shape) == (7,) and tuple(m.noise.shape) == (7,)
        assert torch.equal(m.bias.detach(), torch.zeros(7))
        s = Fnn.softplus(m.noise.detach().double())
        assert torch.allclose(s, torch.ones(7, dtype=torch.float64), rtol=0, atol=1e-7)
        assert not m.clamp_loadings


def test_training_loops_clamp_only_non_negative_loadings():
    import gpzoo_b200 as gz
    from gpzoo_b200.utilities import _clamped
    y = torch.poisson(torch.full((7, 30), 2.0))
    gp = gz.gp.SVGP(gz.kernels.NSF_RBF(L=3), dim=2, M=8)
    nsf = gz.likelihoods.NSF2(gp, y, L=3)
    assert list(_clamped(nsf, ("W",))) == [nsf.W]
    for cls, prior, kw in _models(y):
        assert list(_clamped(cls(prior, y, **kw), ("W", "W2"))) == []


def test_sparse_counts_raise_not_implemented():
    import gpzoo_b200 as gz
    y = torch.poisson(torch.full((7, 30), 2.0))
    ys = SparseCounts.from_dense(y)
    m = gz.likelihoods.FA(gz.gp.GaussianPrior(y, L=2), ys, L=2)
    with pytest.raises(NotImplementedError, match="to_dense"):
        m.elbo(ys)


def test_cpu_tensors_raise_gpz_error():
    import gpzoo_b200 as gz
    from gpzoo_b200 import _cabi
    _lib()
    y = torch.randn(7, 30)
    m = gz.likelihoods.FA(gz.gp.GaussianPrior(y, L=2), y, L=2)
    with pytest.raises(_cabi.GpzError):
        m.elbo(y)


def test_closed_form_is_the_monte_carlo_limit():
    """The closed form equals the Monte-Carlo mean of Normal(bias + W F_e, s).log_prob(y).sum() over E draws of F within four
    standard errors, with variance-mode factors (some below the clamp) and std-dev-mode factors."""
    g = torch.Generator().manual_seed(0)
    G, N, F, nv, cm, E = 6, 9, 4, 2, 0.05, 40000
    dt = torch.float64
    W, bias = torch.randn(G, F, generator=g, dtype=dt), torch.randn(G, generator=g, dtype=dt)
    noise = torch.randn(G, generator=g, dtype=dt)
    mean = torch.randn(F, N, generator=g, dtype=dt)
    spread = 0.05 + 0.5 * torch.rand(F, N, generator=g, dtype=dt)
    spread[0, :3] = 1e-3                                          # below the variance clamp
    y = torch.randn(G, N, generator=g, dtype=dt)
    ref = closed_form(y, W, bias, noise, mean, spread, nv, cm)
    sd = torch.cat((spread[:nv].clamp(min=cm).sqrt(), spread[nv:]), 0)
    Fs = mean + sd * torch.randn(E, F, N, generator=g, dtype=dt)
    pY = torch.distributions.Normal(bias[:, None] + W @ Fs, Fnn.softplus(noise)[:, None])
    per_draw = pY.log_prob(y).sum((1, 2))
    se = per_draw.std() / math.sqrt(E)
    assert abs(float(per_draw.mean() - ref)) <= 4 * float(se), (float(per_draw.mean()), float(ref), float(se))
