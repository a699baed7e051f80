"""Observation models with GPzoo's `gpzoo.likelihoods` surface (likelihoods.py:7-374).

Two ways to use them:

* `model(X, E)` / `model.forward_batched(X, idx, E)` return the same tuples of torch distributions as the
  reference (`pY, qF, qU, pU[, qF2, pF2]`), so existing training loops (`pY.log_prob(y)`,
  `kl_divergence(qU, pU)`) run unchanged.  This compatibility path has to materialise `pY.rate` (E x G x N).
* `model.elbo(X, y, ...)` is the fused hot path: GP moments -> one Poisson likelihood kernel that reads y once and
  returns the log-likelihood and all its gradients -> fused KL.  Nothing of size G x N is written.
  `utilities.train*` use it.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn
from torch import distributions

from . import functional as F


def _sample(qF, E, eps=None):
    """qF.rsample((E,)) (torch normal.py) with an optional externally supplied standard-normal draw."""
    if eps is None:
        return qF.rsample((E,))
    return qF.loc + eps * qF.scale


def _kl_of(m):
    """Per-factor KL(qU || pU) of a `moments` result: the fused chain's own output when it ran, else the KL kernel."""
    return m["kl"] if m.get("kl") is not None else F.MvnKL.apply(m["T"], m["q"], m["Lc"], m["Lu"])


def _gp_moments(gp, X, idx, kwargs):
    """The fused ELBOs' GP moments at the minibatch X[idx], with the multi-group labels `groupsX` when given (their KL: `_kl_of`)."""
    Xb = X if idx is None else X[idx]
    gX = kwargs.get("groupsX")
    return gp.moments(Xb, gX) if gX is not None else gp.moments(Xb)


def _gp_call(gp, X, verbose, kwargs):
    # keywords, as the reference calls its priors (likelihoods.py:81, 111): MGGP_SVGP.forward(X, groupsX, verbose) and
    # MGGP_WSVGP.forward(X, verbose, **args) both take groupsX by name
    return gp(X, verbose=verbose, **kwargs)


# ------------------------------------------------------------------------------------------------
# Gaussian
# ------------------------------------------------------------------------------------------------
class GaussianLikelihood(nn.Module):
    """pY = Normal(F, softplus(noise)), F ~ qF (likelihoods.py:7-20)."""

    def __init__(self, gp, noise=0.1):
        super().__init__()
        self.gp = gp
        self.noise = nn.Parameter(torch.tensor(noise))

    def forward(self, X, E=1, verbose=False, eps=None, **kwargs):
        qF, qU, pU = _gp_call(self.gp, X, verbose, kwargs)
        Fs = _sample(qF, E, eps)
        noise = torch.nn.functional.softplus(self.noise)
        return distributions.Normal(Fs, noise, validate_args=False), qF, qU, pU

    def elbo(self, X, y, E=1, eps=None, **kwargs):
        """mean_E sum_n log N(y | F, noise) - sum KL (utilities.py:479-481).  The likelihood term is O(E*N)
        element-wise work on top of the fused GP moments and stays in torch."""
        pY, _, qU, pU = self.forward(X, E=E, eps=eps, **kwargs)
        return pY.log_prob(y).mean(0).sum() - distributions.kl_divergence(qU, pU).sum()


class ExactLikelihood(nn.Module):
    """pY = Normal(qF.mean, softplus(noise)) (likelihoods.py:23-36)."""

    def __init__(self, gp, noise=0.1):
        super().__init__()
        self.gp = gp
        self.noise = nn.Parameter(torch.tensor(noise))

    def forward(self, X, E=1, verbose=False, **kwargs):
        qF, qU, pU = _gp_call(self.gp, X, verbose, kwargs)
        noise = torch.nn.functional.softplus(self.noise)
        return distributions.Normal(qF.mean, noise, validate_args=False), qF, qU, pU


# ------------------------------------------------------------------------------------------------
# Poisson family
# ------------------------------------------------------------------------------------------------
class _PoissonCounts:
    """The count model of the Poisson family: the fused likelihood call of `elbo` and the distribution `forward` returns.
    The negative-binomial models override both (`_NegBinCounts`)."""

    def _count_ll(self, y, idx, W, V, *args):
        return F.PoissonLL.apply(y, idx, W, V, *args)

    def _pY(self, rate):
        return _poisson(rate)


class PoissonFactorization(_PoissonCounts, nn.Module):
    """Base of PNMF / NSF2: loadings W (G x L), rate contraction softplus(W) @ exp(F) (likelihoods.py:39-53)."""

    _w_softplus = True

    def __init__(self, prior, y, L=10):
        super().__init__()
        D, N = y.shape
        self.prior = prior
        self.W = nn.Parameter(torch.rand((D, L)))

    def get_rate(self, prior_samples):
        """E x G x N un-scaled rate (V = 0 softplus'd to log 2 is NOT applied here, as in the reference)."""
        E, _, B = prior_samples.shape
        ones = None
        # rate kernel multiplies by softplus(V); feed V with softplus(V) = 1  ->  V = log(e - 1)
        v = torch.full((B,), 0.5413248546129181, dtype=prior_samples.dtype, device=prior_samples.device)
        return F.poisson_rate(self.W.to(prior_samples.dtype), v, ones, prior_samples, self._w_softplus)


def _poisson(rate):
    return distributions.Poisson(rate, validate_args=False)


class _FusedPoissonMixin(_PoissonCounts):
    """Fused ELBO for models with one SVGP-family prior (NSF2 / NSF / MGGP_NSF)."""

    def _gp(self):
        return self.prior if hasattr(self, "prior") else self.gp

    def elbo(self, X, y, idx=None, E=1, eps=None, with_lgamma=True, return_parts=False, kl_weight=1.0, **kwargs):
        """ELBO = mean_E sum log p(y | F) - sum_l KL(qU_l || pU_l)   (utilities.py:479-481, 611-616).

        X: N x D (all spots); idx: optional minibatch indices (as forward_batched); y: G x N;
        eps: optional E x L x B standard-normal draw (else drawn from the global RNG on the device);
        kl_weight: data-parallel ranks pass 1/world_size so that the all-reduced sum counts the KL once."""
        gp = self._gp()
        m = _gp_moments(gp, X, idx, kwargs)
        mean, var = m["mean"], m["var"]
        if eps is None:
            eps = torch.randn((E,) + tuple(mean.shape), dtype=mean.dtype, device=mean.device)
        W = self.W.to(mean.dtype)
        ll = self._count_ll(y, idx, W, self.V.to(mean.dtype), mean, var, eps, mean.shape[0], gp.clamp_min, self._w_softplus,
                            with_lgamma)
        kl = _kl_of(m).to(mean.dtype)
        out = ll - kl_weight * kl.sum()
        if return_parts:
            return out, dict(ll=ll, kl=kl, mean=mean, var=var)
        return out


class PNMF(PoissonFactorization):
    """Non-spatial Poisson NMF with a GaussianPrior (likelihoods.py:56-72)."""

    def __init__(self, prior, y, L=10):
        super().__init__(prior=prior, y=y, L=L)
        D, N = y.shape
        self.V = nn.Parameter(torch.ones((N,)))
        self.X = nn.Parameter(torch.zeros((N, 2)), requires_grad=False)

    def forward(self, E=10, eps=None, **kwargs):
        qF, pF = self.prior()
        Fs = _sample(qF, E, eps)
        rate = F.poisson_rate(self.W, self.V, None, Fs, True)
        return self._pY(rate), qF, pF

    def elbo(self, y, idx=None, E=10, eps=None, with_lgamma=True):
        """mean_E sum log p(y|F) - sum KL(qF || pF), fused likelihood kernel (sd-mode factors)."""
        qF, pF = self.prior() if idx is None else self.prior.forward_batched(idx)
        if eps is None:
            eps = torch.randn((E,) + tuple(qF.loc.shape), dtype=qF.loc.dtype, device=qF.loc.device)
        ll = self._count_ll(y, idx, self.W, self.V, qF.loc, qF.scale, eps, 0, 0.0, True, with_lgamma)
        return ll - distributions.kl_divergence(qF, pF).sum()


class NSF2(_FusedPoissonMixin, PoissonFactorization):
    """Non-negative spatial factorisation, softplus loadings (likelihoods.py:74-97)."""

    def __init__(self, gp, y, L=10):
        super().__init__(prior=gp, y=y, L=L)
        D, N = y.shape
        self.V = nn.Parameter(torch.ones((N,)))

    def forward(self, X, E=10, verbose=False, eps=None, **kwargs):
        qF, qU, pU = _gp_call(self.prior, X, verbose, kwargs)
        Fs = _sample(qF, E, eps)
        rate = F.poisson_rate(self.W.to(Fs.dtype), self.V.to(Fs.dtype), None, Fs, True)
        return self._pY(rate), qF, qU, pU

    def forward_batched(self, X, idx, E=10, verbose=False, eps=None, **kwargs):
        qF, qU, pU = _gp_call(self.prior, X[idx], verbose, kwargs)
        Fs = _sample(qF, E, eps)
        rate = F.poisson_rate(self.W.to(Fs.dtype), self.V.to(Fs.dtype), idx, Fs, True)
        return self._pY(rate), qF, qU, pU


class NSF(_FusedPoissonMixin, nn.Module):
    """Older single-module NSF (likelihoods.py:213-253); attribute is `gp`, not `prior`."""

    _w_softplus = True

    def __init__(self, gp, y, L=10):
        super().__init__()
        D, N = y.shape
        self.gp = gp
        self.W = nn.Parameter(torch.rand((D, L)))
        self.V = nn.Parameter(torch.ones((N,)))

    def forward(self, X, E=10, verbose=False, eps=None, **kwargs):
        qF, qU, pU = _gp_call(self.gp, X, verbose, kwargs)
        Fs = _sample(qF, E, eps)
        return _poisson(F.poisson_rate(self.W, self.V, None, Fs, self._w_softplus)), qF, qU, pU

    def forward_batched(self, X, idx, E=10, verbose=False, eps=None, **kwargs):
        qF, qU, pU = _gp_call(self.gp, X[idx], verbose, kwargs)
        Fs = _sample(qF, E, eps)
        return _poisson(F.poisson_rate(self.W, self.V, idx, Fs, self._w_softplus)), qF, qU, pU


class MGGP_NSF(NSF):
    """NSF over an MGGP_SVGP with positional group labels (likelihoods.py:335-374)."""

    def forward(self, X, groupsX, E=10, verbose=False, eps=None):
        return super().forward(X, E=E, verbose=verbose, eps=eps, groupsX=groupsX)

    def forward_batched(self, X, groupsX, idx, E=10, verbose=False, eps=None):
        return super().forward_batched(X, idx, E=E, verbose=verbose, eps=eps, groupsX=groupsX[idx])


class Hybrid_NSF2(_PoissonCounts, nn.Module):
    """Spatial (GP) + non-spatial (GaussianPrior) factors (likelihoods.py:100-163)."""

    def __init__(self, gp, prior, y, L=10, T=10):
        super().__init__()
        D, N = y.shape
        self.sf = PoissonFactorization(prior=gp, y=y, L=L)
        self.cf = PoissonFactorization(prior=prior, y=y, L=T)
        self.V = nn.Parameter(torch.ones((N,)))

    def _combine(self, qF1, qF2, idx, E, eps, eps2):
        F1 = _sample(qF1, E, eps)
        F2 = _sample(qF2, E, eps2)
        Fs = torch.cat((F1, F2), dim=1)
        W = torch.cat((self.sf.W, self.cf.W), dim=1).to(Fs.dtype)
        return self._pY(F.poisson_rate(W, self.V.to(Fs.dtype), idx, Fs, True))

    def forward(self, X, E=10, verbose=False, eps=None, eps2=None, **kwargs):
        qF1, qU, pU = _gp_call(self.sf.prior, X, verbose, kwargs)
        qF2, pF2 = self.cf.prior()
        return self._combine(qF1, qF2, None, E, eps, eps2), qF1, qU, pU, qF2, pF2

    def forward_batched(self, X, idx, E=10, verbose=False, eps=None, eps2=None, **kwargs):
        qF1, qU, pU = _gp_call(self.sf.prior, X[idx], verbose, kwargs)
        qF2, pF2 = self.cf.prior.forward_batched(idx)
        return self._combine(qF1, qF2, idx, E, eps, eps2), qF1, qU, pU, qF2, pF2

    def forward_precomputed(self, W, idx, E=10, verbose=False, eps=None, eps2=None, **kwargs):
        """likelihoods.py:147-163: the spatial prior evaluated from a precomputed W = Kxz Lc^-T (whitened GPs only)."""
        qF1, qU, pU = self.sf.prior.forward_precomputed(W, verbose=verbose, **kwargs)
        qF2, pF2 = self.cf.prior.forward_batched(idx)
        return self._combine(qF1, qF2, idx, E, eps, eps2), qF1, qU, pU, qF2, pF2

    def elbo(self, X, y, idx=None, E=1, eps=None, eps2=None, with_lgamma=True, kl_weight=1.0, **kwargs):
        """Fused hybrid ELBO: ll - sum KL(qU||pU) - sum KL(qF2||pF2)   (utilities.py:509-516).
        The L spatial factors enter the likelihood kernel as (mean, variance), the T non-spatial ones as
        (mean, sd); both loading blocks are contracted in the same pass over y."""
        gp = self.sf.prior
        Xb = X if idx is None else X[idx]
        gX = kwargs.get("groupsX")
        m = gp.moments(Xb, gX) if gX is not None else gp.moments(Xb)
        qF2, pF2 = self.cf.prior() if idx is None else self.cf.prior.forward_batched(idx)
        mean1, var1 = m["mean"], m["var"]
        dt, dev = mean1.dtype, mean1.device
        L, T = mean1.shape[0], qF2.loc.shape[0]
        B = mean1.shape[1]
        if eps is None:
            eps = torch.randn((E, L, B), dtype=dt, device=dev)
        if eps2 is None:
            eps2 = torch.randn((E, T, B), dtype=dt, device=dev)
        mean = torch.cat((mean1, qF2.loc.to(dt)), 0)
        spread = torch.cat((var1, qF2.scale.to(dt)), 0)
        W = torch.cat((self.sf.W, self.cf.W), dim=1).to(dt)
        ll = self._count_ll(y, idx, W, self.V.to(dt), mean, spread, torch.cat((eps, eps2), 1), L, gp.clamp_min, True, with_lgamma)
        kl = _kl_of(m).to(dt)
        return ll - kl_weight * kl.sum() - distributions.kl_divergence(qF2, pF2).sum()


class Hybrid_NSF_Exact(Hybrid_NSF2):
    """Sampling replaced by the log-normal mean, F = mean + var/2 (likelihoods.py:167-210)."""

    def _combine(self, qF1, qF2, idx, E, eps, eps2):
        F1 = (qF1.mean + 0.5 * qF1.scale ** 2).unsqueeze(0)
        F2 = (qF2.mean + 0.5 * qF2.scale ** 2).unsqueeze(0)
        Fs = torch.cat((F1, F2), dim=1)
        W = torch.cat((self.sf.W, self.cf.W), dim=1).to(Fs.dtype)
        return _poisson(F.poisson_rate(W, self.V.to(Fs.dtype), idx, Fs, True)[0])


class Hybrid_NSF(NSF):
    """Older hybrid with RAW (un-softplussed) loadings W | W2, kept non-negative by the training loop's clamp
    (likelihoods.py:281-330; utilities.py:523-524)."""

    _w_softplus = False

    def __init__(self, gp, y, L=10, non_spatial_factors=10):
        super().__init__(gp=gp, y=y, L=L)
        D, N = y.shape
        self.W2 = nn.Parameter(torch.rand((D, non_spatial_factors)))
        self.mF = nn.Parameter(torch.zeros((non_spatial_factors, N)))
        self.scale_qF = nn.Parameter(1e-1 * torch.rand((non_spatial_factors, N)))

    def _q2(self, idx):
        s = torch.nn.functional.softplus(self.scale_qF)
        m = self.mF
        if idx is not None:
            s, m = s[:, idx], m[:, idx]
        return (distributions.Normal(m, s, validate_args=False),
                distributions.Normal(torch.zeros_like(m), torch.ones_like(s), validate_args=False))

    def _run(self, X, idx, E, verbose, eps, eps2, kwargs):
        qF, qU, pU = _gp_call(self.gp, X if idx is None else X[idx], verbose, kwargs)
        qF2, pF2 = self._q2(idx)
        Fs = torch.cat((_sample(qF, E, eps), _sample(qF2, E, eps2)), dim=1)
        W = torch.cat((self.W, self.W2), dim=1).to(Fs.dtype)
        return _poisson(F.poisson_rate(W, self.V.to(Fs.dtype), idx, Fs, False)), qF, qU, pU, qF2, pF2

    def forward(self, X, E=10, verbose=False, eps=None, eps2=None, **kwargs):
        return self._run(X, None, E, verbose, eps, eps2, kwargs)

    def forward_batched(self, X, idx, E=10, verbose=False, eps=None, eps2=None, **kwargs):
        return self._run(X, idx, E, verbose, eps, eps2, kwargs)

    def elbo(self, X, y, idx=None, E=1, eps=None, eps2=None, with_lgamma=True, kl_weight=1.0, **kwargs):
        """Fused ELBO of the raw-loading hybrid (utilities.py:498-529): ll - sum KL(qU||pU) - sum KL(qF2||pF2)."""
        gp = self.gp
        Xb = X if idx is None else X[idx]
        gX = kwargs.get("groupsX")
        m = gp.moments(Xb, gX) if gX is not None else gp.moments(Xb)
        qF2, pF2 = self._q2(idx)
        mean1, var1 = m["mean"], m["var"]
        dt, dev = mean1.dtype, mean1.device
        L, T2, B = mean1.shape[0], qF2.loc.shape[0], mean1.shape[1]
        eps = torch.randn((E, L, B), dtype=dt, device=dev) if eps is None else eps
        eps2 = torch.randn((E, T2, B), dtype=dt, device=dev) if eps2 is None else eps2
        W = torch.cat((self.W, self.W2), dim=1).to(dt)
        ll = F.PoissonLL.apply(y, idx, W, self.V.to(dt), torch.cat((mean1, qF2.loc.to(dt)), 0),
                               torch.cat((var1, qF2.scale.to(dt)), 0), torch.cat((eps, eps2), 1), L, gp.clamp_min, False,
                               with_lgamma)
        kl = _kl_of(m).to(dt)
        return ll - kl_weight * kl.sum() - distributions.kl_divergence(qF2, pF2).sum()


# ------------------------------------------------------------------------------------------------
# Negative binomial: the Poisson models with one dispersion per gene
# ------------------------------------------------------------------------------------------------
class _NegBinCounts:
    """NB(y | r, theta_g) with theta = softplus(dispersion) (G, initialised to log(e - 1): theta = 1) in place of Poisson(r):
    `elbo` runs the fused K7-NB call (functional.NegBinLL), `forward` returns
    NegativeBinomial(total_count=theta[:, None], logits=log r - log theta[:, None]), whose mean is r.  In data-parallel training
    `dispersion` is a shared gradient like W: include it in distributed.FlatGradReducer's list."""

    def _init_dispersion(self, G):
        self.dispersion = nn.Parameter(torch.full((G,), math.log(math.e - 1.0)))

    def _count_ll(self, y, idx, W, V, *args):
        return F.NegBinLL.apply(y, idx, W, V, self.dispersion.to(W.dtype), *args)      # SparseCounts: NotImplementedError

    def _pY(self, rate):
        theta = torch.nn.functional.softplus(self.dispersion.to(rate.dtype))[:, None]
        return distributions.NegativeBinomial(total_count=theta, logits=rate.log() - theta.log(), validate_args=False)


class NSF2_NB(_NegBinCounts, NSF2):
    """NSF2 with a negative-binomial likelihood: any prior NSF2 takes (SVGP, VNNGP, MGGP_SVGP with groupsX, WSVGP)."""

    def __init__(self, gp, y, L=10):
        super().__init__(gp, y, L=L)
        self._init_dispersion(y.shape[0])


class PNMF_NB(_NegBinCounts, PNMF):
    """PNMF with a negative-binomial likelihood."""

    def __init__(self, prior, y, L=10):
        super().__init__(prior, y, L=L)
        self._init_dispersion(y.shape[0])


class Hybrid_NSF2_NB(_NegBinCounts, Hybrid_NSF2):
    """Hybrid_NSF2 with a negative-binomial likelihood."""

    def __init__(self, gp, prior, y, L=10, T=10):
        super().__init__(gp, prior, y, L=L, T=T)
        self._init_dispersion(y.shape[0])


# ------------------------------------------------------------------------------------------------
# Gaussian factor models: real-valued loadings, one noise and one intercept per gene
# ------------------------------------------------------------------------------------------------
class _GaussianFactors:
    """y_g ~ N(bias_g + W_g F, s_g^2), s = softplus(noise) (G; initialised to log(e - 1): s = 1), W real (G x L, torch.randn), bias
    zeros (G).  `elbo` runs the fused K7-G call (functional.GaussianLL), whose expectation over q(F) is exact: it draws no samples.
    The loadings are real, so the training loops do not clamp them (`clamp_loadings`).  In data-parallel training W, bias and
    noise are shared gradients: include model.W, model.bias, model.noise in distributed.FlatGradReducer's list."""

    clamp_loadings = False

    def _init_params(self, G, L):
        self.W = nn.Parameter(torch.randn((G, L)))
        self.bias = nn.Parameter(torch.zeros(G))            # not data-dependent: every data-parallel rank starts from the same value
        self.noise = nn.Parameter(torch.full((G,), math.log(math.e - 1.0)))

    def _ll(self, y, idx, mean, spread, n_var, clamp_min):
        dt = mean.dtype
        return F.GaussianLL.apply(y, idx, self.W.to(dt), self.bias.to(dt), self.noise.to(dt), mean, spread, n_var, clamp_min)

    def _pY(self, Fs):
        """Normal(bias + W F_e, s) over the E x G x B loc, materialised on the library's GEMM (compatibility path)."""
        dt = Fs.dtype
        loc = F.matmul(self.W.to(dt), Fs.contiguous()) + self.bias.to(dt)[:, None]
        scale = torch.nn.functional.softplus(self.noise.to(dt))[:, None]
        return distributions.Normal(loc, scale, validate_args=False)


class RSF(_GaussianFactors, nn.Module):
    """Real-valued spatial factorization: GP factors with real loadings and a Gaussian likelihood with one noise per gene.
    Takes every prior NSF2 takes (SVGP, VNNGP, MGGP_SVGP with groupsX, WSVGP)."""

    def __init__(self, gp, y, L=10):
        super().__init__()
        G, N = y.shape
        self.prior = gp
        self._init_params(G, L)

    def elbo(self, X, y, idx=None, E=1, eps=None, kl_weight=1.0, return_parts=False, **kwargs):
        """ELBO = sum_{g,n} E_q[log N(y | bias + W F, s^2)] - kl_weight sum_l KL(qU_l || pU_l), the expectation in closed form.

        X: N x D (all spots); idx: optional minibatch indices; y: G x N real values (dense).  E and eps are accepted so that the
        training loops can call it, and ignored: no samples are drawn.  kl_weight: data-parallel ranks pass 1/world_size."""
        gp = self.prior
        m = _gp_moments(gp, X, idx, kwargs)
        mean, var = m["mean"], m["var"]
        ll = self._ll(y, idx, mean, var, mean.shape[0], gp.clamp_min)
        kl = _kl_of(m).to(mean.dtype)
        out = ll - kl_weight * kl.sum()
        if return_parts:
            return out, dict(ll=ll, kl=kl, mean=mean, var=var)
        return out

    def forward(self, X, E=10, verbose=False, eps=None, **kwargs):
        qF, qU, pU = _gp_call(self.prior, X, verbose, kwargs)
        return self._pY(_sample(qF, E, eps)), qF, qU, pU

    def forward_batched(self, X, idx, E=10, verbose=False, eps=None, **kwargs):
        qF, qU, pU = _gp_call(self.prior, X[idx], verbose, kwargs)
        return self._pY(_sample(qF, E, eps)), qF, qU, pU


class FA(_GaussianFactors, nn.Module):
    """Factor analysis: non-spatial factors (a GaussianPrior) with real loadings and one noise per gene."""

    def __init__(self, prior, y, L=10):
        super().__init__()
        G, N = y.shape
        self.prior = prior
        self._init_params(G, L)

    def elbo(self, y, idx=None, E=10, eps=None, **kwargs):
        """sum_{g,n} E_q[log N(y | bias + W F, s^2)] - sum KL(qF || pF), the expectation in closed form (E and eps are ignored)."""
        qF, pF = self.prior() if idx is None else self.prior.forward_batched(idx)
        ll = self._ll(y, idx, qF.loc, qF.scale, 0, 0.0)
        return ll - distributions.kl_divergence(qF, pF).sum()

    def forward(self, E=10, eps=None, **kwargs):
        qF, pF = self.prior()
        return self._pY(_sample(qF, E, eps)), qF, pF
