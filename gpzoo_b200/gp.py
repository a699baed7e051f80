"""Sparse GP modules with GPzoo's `gpzoo.gp` surface (SVGP, MGGP_SVGP, WSVGP, MGGP_WSVGP, VNNGP,
GaussianPrior) on top of the fused CUDA kernels.

Constructor arguments, parameter names/shapes (`Z`, `Lu`, `mu`, `groupsZ`), the `jitter`/`K` attributes and
the returned `(qF, qU, pU)` distributions follow the reference (gp.py:7-399).  Users overwrite the
parameters after construction (scalar GP -> L-batched, SURVEY.md §5), so shapes are resolved at call time.

Inside `forward` the reference's chain cholesky -> cholesky_solve -> Lu Lu^T -> svgp_forward is replaced by
CholeskyInverse -> Whiten -> Predict (functional.py); `kl_divergence(qU, pU)` on the returned distributions
dispatches to the fused KL kernel through `register_kl`.
"""
from __future__ import annotations

import torch
import torch.nn as nn
from torch import distributions
from torch.distributions import constraints
from torch.distributions.kl import register_kl

from . import functional as F


class VariationalMVN(distributions.MultivariateNormal):
    """qU = N(mu, Lu Lu^T) carrying the whitened factors so that KL(qU || pU) needs no further solves."""

    def __init__(self, loc, scale_tril, gpz_state):
        super().__init__(loc, scale_tril=scale_tril, validate_args=False)
        self._gpz_state = gpz_state          # (T, q, Lc, Lu) L-batched tensors, batched flag, per-factor KL if already computed


class PriorMVN(distributions.MultivariateNormal):
    """pU = N(0, Lc Lc^T)."""

    def __init__(self, loc, scale_tril):
        super().__init__(loc, scale_tril=scale_tril, validate_args=False)


@register_kl(VariationalMVN, PriorMVN)
def _kl_variational_prior(qU, pU):
    T, q, Lc, Lu, batched, kl = qU._gpz_state
    kl = (kl if kl is not None else F.MvnKL.apply(T, q, Lc, Lu)).to(qU.loc.dtype)
    return kl if batched else kl[0]


def _as3(t):
    return t if t.dim() == 3 else t.unsqueeze(0)


class _SparseGPBase(nn.Module):
    clamp_min = 1e-6

    def _init_params(self, kernel, dim, M, jitter):
        self.kernel = kernel
        self.jitter = jitter
        self.Z = nn.Parameter(torch.randn((M, dim)))
        self.Lu = nn.Parameter(torch.randn((M, M)))
        self.mu = nn.Parameter(torch.zeros((M,)))
        self.constraint = constraints.lower_cholesky

    # -- kernel calls -------------------------------------------------------------------------------
    def _kernel_matrices(self, X, groupsX=None, want_lo=False, want_h=False, skip_kzz=False, skip_kzx=False):
        """Kxx (diag), Kzx, Kzz (+jitter).  want_lo: Kzx comes back as (Kzx, Kzx_lo) for the split-TF32 tensor-core path;
        want_h: as (stand-in, Kh, Kl, scale) fp16 planes for the split-FP16 path.  skip_*: leave that matrix out (None)."""
        kw = {"_want_h": True} if want_h else ({"_want_lo": True} if want_lo else {})
        Kxx = Kzx = Kzz = None
        if groupsX is not None:
            gZ = self.groupsZ
            if not skip_kzx:
                Kxx = self.kernel(X, X, groupsX, groupsX, diag=True)
                Kzx = self.kernel(self.Z, X, gZ, groupsX, **kw)
            if not skip_kzz:
                Kzz = self.kernel(self.Z, self.Z, gZ, gZ, _jitter=self.jitter)      # add_jitter fused (gp.py:209/360)
        else:
            if not skip_kzx:
                Kxx = self.kernel(X, X, diag=True)
                Kzx = self.kernel(self.Z, X, **kw)
            if not skip_kzz:
                Kzz = self.kernel(self.Z, self.Z, _jitter=self.jitter)
        return Kxx, Kzx, Kzz

    def _whitened(self, Kzz, consume=False):
        """Lc, Linv, Lu, T, q with a common leading L.  consume: Kzz is a temporary of the caller and may be overwritten.
        Leaves the per-factor KL in `self._chain_kl` when the fused chain computed it (None otherwise)."""
        Kzz = _as3(Kzz)
        mu = self.mu if self.mu.dim() == 2 else self.mu.unsqueeze(0)
        Lu_raw = _as3(self.Lu)
        L = max(Kzz.shape[0], mu.shape[0], Lu_raw.shape[0])
        self._chain_kl = None
        if Kzz.shape[0] == L and F.chain_ok(Kzz.dtype, Kzz.shape[-1]):
            ex = lambda t: t if t.shape[0] == L else t.expand(L, *t.shape[1:])
            Lc, Linv, Lu, T, q, kl = F.SvgpChain.apply(Kzz, ex(Lu_raw.to(Kzz.dtype)), ex(mu.to(Kzz.dtype)), bool(consume))
            self._chain_kl = kl
            return Lc, Linv, Lu, T, q, L
        Lc, Linv = F.CholeskyInverse.apply(Kzz)
        if Lc.shape[0] != L:
            Lc, Linv = Lc.expand(L, -1, -1), Linv.expand(L, -1, -1)
        Lu = F.LowerCholesky.apply(Lu_raw.to(Kzz.dtype))
        if Lu.shape[0] != L:
            Lu = Lu.expand(L, -1, -1)
        if mu.shape[0] != L:
            mu = mu.expand(L, -1)
        T, q = F.Whiten.apply(Linv, Lu, mu.to(Kzz.dtype))
        return Lc, Linv, Lu, T, q, L

    def _chain_dtype(self, dt):
        """Arithmetic of the O(M^3) chain (Kzz build, Cholesky + inverse, whitening, KL and their backward).  The chain is where
        the conditioning of Kzz enters (its fp32 error grows like cond(Kzz) * 6e-8, for the reference's fp32 too), and up to
        M = F.CHAIN_FP64_MAX_M it is latency-bound and costs the same in double precision: fp32 models run it in fp64 there
        and hand fp32 Linv / T / q to the N-proportional kernels.  Above that size it runs in the model's dtype."""
        if dt == torch.float32 and self.Z.shape[0] <= F.CHAIN_FP64_MAX_M:
            return torch.float64
        return dt

    def _kzz(self, X, groupsX, cdt):
        if cdt == X.dtype:
            return self._kernel_matrices(X, groupsX, skip_kzx=True)[2]
        Zc = self.Z.to(cdt)
        if groupsX is not None:
            return self.kernel(Zc, Zc, self.groupsZ, self.groupsZ, _jitter=self.jitter)
        return self.kernel(Zc, Zc, _jitter=self.jitter)

    _fusable = True          # SVGP / MGGP_SVGP: chain + predict as ONE autograd node (functional.SvgpMomentsH)

    def _fused_moments(self, X, groupsX, cdt, Kxx, Kzx, side, main):
        """The one-node path (merged backward) when it applies: fp32 chain, M large enough for the fused chain, L-batched
        kernel and variational parameters, autograd on.  Returns the `moments` dict or None."""
        dt = X.dtype
        M = self.Z.shape[0]
        if not (self._fusable and torch.is_grad_enabled() and cdt == dt and F.fused_moments_ok(dt, M, X.shape[0])):
            return None
        mu = self.mu if self.mu.dim() == 2 else self.mu.unsqueeze(0)
        Lu_raw = _as3(self.Lu)
        handle, Kh, Kl, sK = Kzx
        L = max(Kh.shape[0], mu.shape[0], Lu_raw.shape[0])
        if not (Kh.shape[0] == L and mu.shape[0] == L and Lu_raw.shape[0] == L):
            return None
        Kzz = _as3(self._kzz(X, groupsX, cdt))
        if Kzz.shape[0] != L:
            return None
        Kxx = Kxx if Kxx.dim() == 2 else Kxx.unsqueeze(0)
        if Kxx.shape[0] != L:
            Kxx = Kxx.expand(L, -1)
        main.wait_stream(side)
        mean, var, kl, Lc, Lu = F.SvgpMomentsH.apply(Kzz, Lu_raw.to(dt), mu.to(dt), Kxx, handle, Kh, Kl, sK, True,
                                                     getattr(handle, "_gpz_box", None))
        return dict(mean=mean, var=var, kl=kl, Lc=Lc, Lu=Lu, T=None, q=None, _chain=None)

    def moments(self, X, groupsX=None, _chain=None):
        """Fused predictive moments: returns dict(mean, var (unclamped), T, q, Lc, Lu), all L-batched (T, q, Lc, Lu in the
        chain's dtype, see `_chain_dtype`).
        _chain: (Lc, Linv, Lu, T, q, L) of an earlier call with the same parameters (tiled prediction reuses the Kzz chain)."""
        if _chain is None:
            F.clear_step_cache()
        dt = X.dtype
        cdt = self._chain_dtype(dt)
        want_h = F.predict_h_ok(dt, self.Z.shape[0], X.shape[0])
        want_lo = (not want_h) and F.tensor_core_predict_ok(dt, self.Z.shape[0], X.shape[0])
        if _chain is not None:
            Kxx, Kzx, _ = self._kernel_matrices(X, groupsX, want_lo, want_h, skip_kzz=True)
            Lc, Linv, Lu, T, q, L = _chain
        elif want_h and F.OVERLAP_KERNEL_BUILD:
            # The Kzz chain (Cholesky + inverse, latency-bound, about half of the SMs) and the HBM-bound Kzx build are
            # independent: the Kzx kernel runs on a side stream and joins before the predictive GEMMs.  It runs under
            # torch.cuda.stream(side), so autograd runs its BACKWARD on the side stream too (the engine replays every node on
            # the stream of its forward and orders producers / consumers across streams).  The planes live in the side stream's
            # allocator pool and are consumed on the main stream; no record_stream is needed (and it would make the allocator
            # churn): a side-pool block is only ever reused by a later side-stream allocation, and the side stream's work of the
            # next step starts with the wait below, i.e. after everything the main stream had queued when the block was freed.
            side, main = F.side_stream(X.device), torch.cuda.current_stream()
            side.wait_stream(main)
            with torch.cuda.stream(side):
                Kxx, Kzx, _ = self._kernel_matrices(X, groupsX, want_lo, want_h, skip_kzz=True)
            fused = self._fused_moments(X, groupsX, cdt, Kxx, Kzx, side, main)
            if fused is not None:
                return fused
            Lc, Linv, Lu, T, q, L = self._whitened(self._kzz(X, groupsX, cdt), consume=True)
            main.wait_stream(side)
        else:
            Kxx, Kzx, _ = self._kernel_matrices(X, groupsX, want_lo, want_h, skip_kzz=True)
            Lc, Linv, Lu, T, q, L = self._whitened(self._kzz(X, groupsX, cdt), consume=True)
        chain = (Lc, Linv, Lu, T, q, L)
        out = dict(T=T, q=q, Lc=Lc, Lu=Lu, _chain=chain)
        if _chain is None and getattr(self, "_chain_kl", None) is not None:
            out["kl"] = self._chain_kl                  # per-factor KL(qU || pU), already computed by the fused chain
        Linv, T, q = Linv.to(dt), T.to(dt), q.to(dt)            # the N-proportional kernels run in the model's dtype
        Kxx = Kxx if Kxx.dim() == 2 else Kxx.unsqueeze(0)
        if Kxx.shape[0] != L:
            Kxx = Kxx.expand(L, -1)
        if want_h:
            Kzx, Kh, Kl, sK = Kzx
            if Kh.shape[0] != L:
                Kzx, Kh, Kl, sK = Kzx.expand(L, -1, -1), Kh.expand(L, -1, -1), Kl.expand(L, -1, -1), sK.expand(L)
            mean, var = F.PredictH.apply(Kxx, Kzx, Linv, T, q, Kh, Kl, sK)
            return dict(out, mean=mean, var=var)
        Kzx_lo = None
        if want_lo:
            Kzx, Kzx_lo = Kzx
        Kzx = _as3(Kzx)
        if Kzx_lo is not None:
            Kzx_lo = _as3(Kzx_lo)
        if Kzx.shape[0] != L:
            Kzx = Kzx.expand(L, -1, -1)
            Kzx_lo = Kzx_lo.expand(L, -1, -1) if Kzx_lo is not None else None
        mean, var = F.Predict.apply(Kxx, Kzx, Linv, T, q, Kzx_lo)
        return dict(out, mean=mean, var=var)

    @torch.no_grad()
    def predict_moments(self, X, groupsX=None, tile=32768):
        """Predictive mean and (unclamped) variance at ALL rows of X, tile by tile and without autograd state, so the
        footprint is one tile's worth of L x M x tile arrays whatever N is (SURVEY.md §8(f) row 3: the reference's notebooks
        move the model to the CPU to evaluate `model.prior(X)` on every spot, Slideseq_NSF_newest_version.ipynb:624).
        The Kzz chain (Cholesky, inverse, whitening) is computed once and reused by every tile.  Returns (mean, var), L x N."""
        means, variances, chain = [], [], None
        for s0 in range(0, X.shape[0], int(tile)):
            gx = groupsX[s0:s0 + tile] if groupsX is not None else None
            m = self.moments(X[s0:s0 + tile].contiguous(), gx) if chain is None else \
                self.moments(X[s0:s0 + tile].contiguous(), gx, _chain=chain)
            chain = m.get("_chain", None)
            means.append(m["mean"])
            variances.append(m["var"])
        if not means:
            raise ValueError("predict_moments needs at least one point")
        return torch.cat(means, dim=1), torch.cat(variances, dim=1)

    def _batched(self):
        return self.mu.dim() == 2 or self.Lu.dim() == 3 or getattr(self.kernel, "_batched", False)

    def _distributions(self, m):
        b = self._batched()
        mean, var = (m["mean"], m["var"]) if b else (m["mean"][0], m["var"][0])
        Lu, Lc = (m["Lu"], m["Lc"]) if b else (m["Lu"][0], m["Lc"][0])
        Lu, Lc = Lu.to(mean.dtype), Lc.to(mean.dtype)            # (the KL below still uses the chain's own precision)
        qF = distributions.Normal(mean, torch.clamp(var, min=self.clamp_min) ** 0.5, validate_args=False)
        mu = self.mu.to(Lu.dtype)
        qU = VariationalMVN(mu, Lu, (m["T"], m["q"], m["Lc"], m["Lu"], b, m.get("kl")))
        pU = PriorMVN(torch.zeros_like(mu), Lc)
        return qF, qU, pU


class SVGP(_SparseGPBase):
    """Titsias/Hensman sparse variational GP (gp.py:149-232)."""
    clamp_min = 1e-6                                   # gp.py:228

    def __init__(self, kernel, dim=1, M=50, jitter=1e-4):
        super().__init__()
        self._init_params(kernel, dim, M, jitter)
        self.precompute_distance = False               # attribute kept (gp.py:157); the method it shadows is dead code

    def kernel_forward(self, X, Z, **args):
        return self.kernel(X, Z, **args)

    def forward_kernels(self, X, Z=None, **args):
        Kxx, Kzx, Kzz = self.kernel(X, X, diag=True), self.kernel(self.Z, X), self.kernel(self.Z, self.Z)
        return Kxx, Kzx, Kzz

    def forward(self, X, verbose=False):
        return self._distributions(self.moments(X))


class MGGP_SVGP(_SparseGPBase):
    """SVGP with a multi-group kernel; owns the inducing points' group labels (gp.py:329-382)."""
    clamp_min = 5e-2                                   # gp.py:378

    def __init__(self, kernel, dim=1, M=50, jitter=1e-4, n_groups=2):
        super().__init__()
        self.kernel = kernel
        self.jitter = jitter
        self.Z = nn.Parameter(torch.randn((M, dim)))
        self.groupsZ = nn.Parameter(torch.randint(0, n_groups, (M,)).type(torch.LongTensor), requires_grad=False)
        self.Lu = nn.Parameter(torch.randn((M, M)))
        self.mu = nn.Parameter(torch.zeros((M,)))
        self.constraint = constraints.lower_cholesky

    def forward(self, X, groupsX, verbose=False):
        return self._distributions(self.moments(X, groupsX))

    def moments(self, X, groupsX=None, _chain=None):
        if groupsX is None:
            raise TypeError("MGGP_SVGP needs groupsX")
        return super().moments(X, groupsX, _chain=_chain)


class WSVGP(_SparseGPBase):
    """Whitened SVGP (gp.py:235-322): u = Lc v with q(v) = N(mu, Lu Lu^T), so W = Kxz Lc^-T, mean = W mu,
    var = (Kxx - sum W^2) + sum (W Lu)^2 and pZ = None (the caller adds `whitened_KL`).  In the notation of `moments` this is
    the same predictive kernel with T := Lu and q := mu (no whitening products), and KL(q(v) || N(0, I)) is the fused KL
    kernel with Lc := I, which is what `model.elbo(...)` subtracts.  The reference clamps (Kxx - sum W^2) at 0 before adding
    the second term (gp.py:287) — a guard against round-off only (the term is >= 0 in exact arithmetic); here the sum is
    formed in one pass and clamped at 0 as a whole."""
    clamp_min = 0.0
    _fusable = False         # T := Lu, q := mu and the KL is against the identity: the two-node path

    def __init__(self, kernel, dim=1, M=50, jitter=1e-4):
        super().__init__()
        self._init_params(kernel, dim, M, jitter)

    def kernel_forward(self, X, Z, **args):
        return self.kernel(X, Z, **args)

    def forward_kernels(self, X, **args):
        return self._kernel_matrices(X, args.get("groupsX"))

    def _whitened(self, Kzz, consume=False):
        self._chain_kl = None
        Kzz = _as3(Kzz)
        mu = self.mu if self.mu.dim() == 2 else self.mu.unsqueeze(0)
        Lu_raw = _as3(self.Lu)
        L = max(Kzz.shape[0], mu.shape[0], Lu_raw.shape[0])
        ex = lambda t: t if t.shape[0] == L else t.expand(L, *t.shape[1:])
        _, Linv = F.CholeskyInverse.apply(Kzz)
        Lu = ex(F.LowerCholesky.apply(Lu_raw.to(Kzz.dtype)))
        eye = torch.eye(Kzz.shape[-1], dtype=Kzz.dtype, device=Kzz.device).expand(L, -1, -1).contiguous()
        return eye, ex(Linv), Lu, Lu, ex(mu.to(Kzz.dtype)), L          # (Lc := I for the KL, Linv, Lu, T := Lu, q := mu)

    def _whitened_distributions(self, mean, var, Lu):
        if not self._batched():
            mean, var, Lu = mean[0], var[0], Lu[0]
        qF = distributions.Normal(mean, torch.clamp(var, min=0.0) ** 0.5, validate_args=False)
        qZ = distributions.MultivariateNormal(self.mu.to(Lu.dtype), scale_tril=Lu, validate_args=False)
        return qF, qZ, None

    def forward(self, X, verbose=False, **args):
        m = self.moments(X, args.get("groupsX"))
        return self._whitened_distributions(m["mean"], m["var"], m["Lu"].to(m["mean"].dtype))

    def forward_precomputed(self, W, **args):
        """gp.py:308-322: predictive distribution from a precomputed W = Kxz Lc^-T (L x N x M), skipping the kernel build and
        the Cholesky.  Kxx is sigma^2 per factor as in the reference ((L,) sigma of the batched kernels; (L,1,1) is accepted
        too).  Runs the fused predictive kernel with A := W^T (the triangular product by Linv := I is the price of reusing it)."""
        W3 = _as3(W)
        L, N, M = W3.shape
        dt = W3.dtype
        mu = self.mu if self.mu.dim() == 2 else self.mu.unsqueeze(0)
        ex = lambda t: t if t.shape[0] == L else t.expand(L, *t.shape[1:])
        Lu = ex(F.LowerCholesky.apply(_as3(self.Lu).to(dt)))
        Kxx = ex((self.kernel.sigma.reshape(-1, 1).to(dt) ** 2)).expand(L, N)
        eye = torch.eye(M, dtype=dt, device=W3.device).expand(L, -1, -1).contiguous()
        mean, var = F.Predict.apply(Kxx, W3.transpose(-2, -1), eye, Lu, ex(mu.to(dt)), None)
        return self._whitened_distributions(mean, var, Lu)


class MGGP_WSVGP(WSVGP):
    """gp.py:385-399: forward(X, groupsX=...) as a keyword (the reference reads args['groupsX'])."""

    def __init__(self, kernel, dim=1, M=50, n_groups=2, jitter=1e-4):
        super().__init__(kernel, dim, M, jitter)
        self.groupsZ = nn.Parameter(torch.randint(0, n_groups, (M,)).type(torch.LongTensor), requires_grad=False)

    def moments(self, X, groupsX=None, _chain=None):
        if groupsX is None:
            raise TypeError("MGGP_WSVGP needs groupsX")
        return super().moments(X, groupsX, _chain=_chain)


class VNNGP(_SparseGPBase):
    """Nearest-neighbour variational GP (gp.py:7-122): each point conditions on its K nearest inducing points only.
    KL(qU || pU) is still the full M-dimensional one (gp.py:119-120).  The reference's unconditional prints
    (gp.py:32,65,79-81,84) are dropped."""
    clamp_min = 5e-2                                   # gp.py:118

    def __init__(self, kernel, dim=1, M=50, K=3, jitter=1e-4):
        super().__init__()
        self.kernel = kernel
        self.jitter = jitter
        self.K = K
        self.Z = nn.Parameter(torch.randn((M, dim)))
        self.Lu = nn.Parameter(torch.randn((M, M)))
        self.mu = nn.Parameter(torch.zeros((M,)))
        self.constraint = constraints.lower_cholesky

    def neighbors(self, X):
        """N x K int64 indices into Z, ascending distance (gp.py:64)."""
        return F.vnngp_neighbors(X, self.Z.to(X.dtype), self.K)

    def moments(self, X, groupsX=None):
        dt = X.dtype
        if getattr(self.kernel, "_ard", False):
            raise NotImplementedError("VNNGP's fused neighbour kernel takes one lengthscale per factor; "
                                      f"{type(self.kernel).__name__} (per-dimension lengthscales) is not supported")
        if getattr(self.kernel, "_kind", 0) != 0:
            raise NotImplementedError("VNNGP's fused neighbour kernel evaluates the RBF cross-covariance; "
                                      f"{type(self.kernel).__name__} is not supported")
        F.clear_step_cache()
        Kzz = _as3(self.kernel(self.Z, self.Z, _jitter=self.jitter))                 # first jitter (gp.py:55)
        Kxx = self.kernel(X, X, diag=True)
        Kxx = Kxx if Kxx.dim() == 2 else Kxx.unsqueeze(0)
        # the full-M chain only feeds KL(qU || pU) (gp.py:119-120) and Lu; it runs in the chain's dtype (fp64 up to M = 256)
        cdt = self._chain_dtype(dt)
        Lc, Linv, Lu_c, T, q, L = self._whitened(Kzz if cdt == dt else self._kzz(X, None, cdt))
        Lu = Lu_c.to(dt)
        if Kzz.shape[0] != L:
            Kzz, Kxx = Kzz.expand(L, -1, -1), Kxx.expand(L, -1)
        S = F.OuterLower.apply(Lu)
        mu = self.mu if self.mu.dim() == 2 else self.mu.unsqueeze(0)
        mu = (mu if mu.shape[0] == L else mu.expand(L, -1)).to(dt)
        sigma = self.kernel.sigma.reshape(-1).to(dt)
        ls = self.kernel.lengthscale.reshape(-1).to(dt)
        if sigma.numel() != L:
            sigma, ls = sigma.expand(L), ls.expand(L)
        nn_idx = self.neighbors(X)
        mean, var = F.VnngpPredict.apply(X, self.Z.to(dt), sigma, ls, Kzz, S, mu, Kxx, nn_idx, float(self.jitter))
        return dict(mean=mean, var=var, T=T, q=q, Lc=Lc, Lu=Lu_c, nn=nn_idx, kl=getattr(self, "_chain_kl", None))

    def forward(self, X, verbose=False):
        return self._distributions(self.moments(X))


class GaussianPrior(nn.Module):
    """Non-spatial mean-field factors (gp.py:125-146): per-spot mean and softplus(scale), prior N(0, scale_pf).
    O(L*N) element-wise parameters; their fused use is inside the Poisson likelihood kernel."""

    def __init__(self, y, L=10):
        super().__init__()
        D, N = y.shape
        self.mean = nn.Parameter(torch.randn(size=(L, N)))
        self.scale = nn.Parameter(torch.rand(size=(L, N)))
        self.scale_pf = 1.0

    def _make(self, mean, scale_raw):
        scale = torch.nn.functional.softplus(scale_raw)
        qF = distributions.Normal(mean, scale, validate_args=False)
        pF = distributions.Normal(torch.zeros_like(mean), self.scale_pf * torch.ones_like(scale), validate_args=False)
        return qF, pF

    def forward(self):
        return self._make(self.mean, self.scale)

    def forward_batched(self, idx):
        return self._make(self.mean[:, idx], self.scale[:, idx])
