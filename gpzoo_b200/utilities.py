"""Hot-path helpers and training loops with GPzoo's `gpzoo.utilities` names.

The functions on or next to the ELBO path (SURVEY.md §2.1 rows 11-13) plus the initialisation pipeline
(`gpzoo_b200.initialisation`, SURVEY §8(f) row 4); the anndata / squidpy / plotting helpers of the
reference (utilities.py:50-69, 86-156, 421-448) are host-side data handling and out of scope (DESIGN.md).  The training loops call the fused `model.elbo(...)`.
"""
from __future__ import annotations

import torch

from . import functional as F
from .kernels import embed_distance_matrix as _embed_distance_matrix  # noqa: F401  (utilities.py:459-469)
# the initialisation pipeline of the notebooks (utilities.py:14-24, 38-44, 71-84, 237-313), on the device
from .initialisation import (build_group_distances, init_softplus, lnormal_approx_dirichlet, regularized_nmf,  # noqa: F401
                             rescale_spatial_coords, shrink_factors, shrink_loadings)


def whitened_KL(mz, Lz):
    """0.5 (-2 sum log diag Lz + |Lz|_F^2 + |mz|^2 - M)   (utilities.py:27-36).

    = KL(N(mz, Lz Lz^T) || N(0, I)): the fused KL kernel with Lc = I (so T = Lz, q = mz).  Accepts a single GP
    (Lz M x M) like the reference, and additionally L-batched inputs (returning one value per factor), for
    which the reference's torch.diagonal call is wrong (SURVEY.md App. B)."""
    single = Lz.dim() == 2
    Lz3 = Lz.unsqueeze(0) if single else Lz
    mz2 = mz.unsqueeze(0) if mz.dim() == 1 else mz
    eye = torch.eye(Lz3.shape[-1], dtype=Lz3.dtype, device=Lz3.device).expand_as(Lz3).contiguous()
    kl = F.MvnKL.apply(Lz3.contiguous(), mz2.contiguous(), eye, Lz3.contiguous())
    return kl[0] if single else kl


def add_jitter(K, jitter=1e-3):
    """In-place diagonal jitter, returns the same tensor (utilities.py:407-418).  The GP modules fuse the jitter
    into the kernel-matrix build instead; this stays for user code."""
    K.diagonal(dim1=-2, dim2=-1).add_(jitter)
    return K


def reshape_param(param):
    """(..., a, b) -> (-1, a, b)   (utilities.py:377-380)."""
    return param.view(-1, param.shape[-2], param.shape[-1])


def svgp_forward(Kxx, Kzz, W, inducing_mean, inducing_cov):
    """mean = W mu (L x N x 1), cov = Kxx + sum_j ((W (S - Kzz)) o W) (L x N)   (utilities.py:382-397), for callers that hold
    W = Kxz Kzz^-1 (L x N x M) already.  Both contractions run on the library's batched GEMM; the GP modules do not come
    through here (they use the fused triangular form, csrc/predict.cu, which needs a third of the flops)."""
    mean = F.matmul(W, inducing_mean.unsqueeze(-1))
    cov = Kxx + (F.matmul(W, inducing_cov - Kzz) * W).sum(-1)
    return mean, cov


def _squared_dist(X, Z):
    """Squared Euclidean distances (utilities.py:399-405).  The reference expands |x|^2 - 2 x.z + |z|^2 and clamps the
    cancellation error at 0; here the differences are formed directly (csrc/kernel_build.cu), so the result is >= 0 by
    construction and exact for coincident points."""
    return F.SquaredDist.apply(X, Z)


def _torch_sqrt(x, eps=1e-12):
    """sqrt(x + eps): the NaN-gradient guard of utilities.py:450-456."""
    return (x + eps).sqrt()


def _step(model, optimizer, elbo_fn, clamp_W):
    optimizer.zero_grad(set_to_none=True)
    loss = -elbo_fn()
    loss.backward()
    optimizer.step()
    with torch.no_grad():
        for w in clamp_W:
            w.clamp_(min=0.0)                      # utilities.py:523-524, 623
    return loss.detach()


def _clamped(model, names):
    """The loadings the loops keep >= 0 after each step (utilities.py:523-524, 623): none for models with real-valued loadings
    (`clamp_loadings = False`: RSF, FA)."""
    if not getattr(model, "clamp_loadings", True):
        return ()
    return [w for w in (getattr(model, n, None) for n in names) if w is not None]


def _finish(losses):
    F.check_cholesky_info()
    return [float(v) for v in torch.stack(losses).cpu()] if losses else []


def train(model, optimizer, X, y, device=None, steps=200, E=20, **kwargs):
    """Full-batch loop (utilities.py:471-493).  The per-step `loss.item()` sync of the reference is replaced
    by one transfer at the end."""
    losses = [_step(model, optimizer, lambda: model.elbo(X, y, E=E, **kwargs), ()) for _ in range(steps)]
    return _finish(losses)


def _sample_idx(N, batch_size, device):
    # utilities.py:605 draws torch.multinomial(ones(N), batch_size) on the CPU; randperm on the device is the
    # same distribution (uniform without replacement) with no host round-trip.
    return torch.randperm(N, device=device)[:batch_size]


def train_batched(model, optimizer, X, y, device=None, steps=200, E=20, batch_size=1000, **kwargs):
    """Minibatch loop (utilities.py:600-631), including the W >= 0 clamp after each update (not for real-valued loadings)."""
    clamp = _clamped(model, ("W",))
    losses = []
    for _ in range(steps):
        idx = _sample_idx(X.shape[0], batch_size, X.device)
        kw = dict(kwargs)
        if "groupsX" in kw:
            kw["groupsX"] = kw["groupsX"][idx]
        losses.append(_step(model, optimizer, lambda: model.elbo(X, y, idx=idx, E=E, **kw), clamp))
    return _finish(losses)


def train_hybrid(model, optimizer, X, y, device=None, steps=200, E=20, **kwargs):
    """utilities.py:531-563 (two KL terms; W, W2 clamped)."""
    ws = _clamped(model, ("W", "W2"))
    losses = [_step(model, optimizer, lambda: model.elbo(X, y, E=E, **kwargs), ws) for _ in range(steps)]
    return _finish(losses)


def train_hybrid_batched(model, optimizer, X, y, device=None, steps=200, E=20, batch_size=1000, **kwargs):
    """utilities.py:498-529; uses the y*log(rate)-rate form of the log-likelihood (utilities.py:507)."""
    ws = _clamped(model, ("W", "W2"))
    losses = []
    for _ in range(steps):
        idx = _sample_idx(X.shape[0], batch_size, X.device)
        losses.append(_step(model, optimizer, lambda: model.elbo(X, y, idx=idx, E=E, with_lgamma=False, **kwargs), ws))
    return _finish(losses)


def train_closure_batched(model, optimizer, X, groupsX, y, device=None, steps=200, E=20, batch_size=1000):
    """Closure-driven minibatch loop of the multi-group models (utilities.py:566-596): `optimizer.step(closure)` with a fresh
    index set per step, for optimisers that re-evaluate the loss (LBFGS).  The closure runs the fused ELBO; the reference's
    debugging prints and its per-evaluation `loss.item()` are dropped (losses are fetched once at the end)."""
    losses = []
    for _ in range(steps):
        idx = _sample_idx(X.shape[0], batch_size, X.device)

        def closure(idx=idx):
            optimizer.zero_grad(set_to_none=True)
            loss = -model.elbo(X, y, idx=idx, E=E, groupsX=groupsX[idx])
            loss.backward()
            losses.append(loss.detach())
            return loss

        optimizer.step(closure)
    return _finish(losses)
