"""Covariance modules with GPzoo's `gpzoo.kernels` surface, computed by the fused CUDA kernel-matrix
build (csrc/kernel_build.cu) instead of torch.cdist + element-wise ops.

Same class names, constructor arguments, parameter names/shapes and call signatures as the reference
(kernels.py:32-228), so model-building code and state_dicts carry over.  Every forward is one launch of
`gpz_kernel_build_fwd_*`; gradients come from `gpz_kernel_build_bwd_*`.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import functional as F


def embed_distance_matrix(distance_matrix):
    """Classical-MDS embedding of a group-distance matrix (init-time helper, utilities.py:459-469).
    Runs once per model in plain torch; its output only feeds the ng x ng r^2 table of the CUDA kernel."""
    D = torch.as_tensor(distance_matrix)
    n = D.shape[0]
    J = torch.eye(n, dtype=D.dtype, device=D.device) - 1.0 / n
    lam, Q = torch.linalg.eigh(-0.5 * (J @ (D * D) @ J))
    return Q * (lam.clamp(min=0) + 1e-6).sqrt()


def _r2_table(embedding, dtype):
    e = embedding.detach().to(dtype)
    d = e[:, None, :] - e[None, :, :]
    return (d * d).sum(-1).contiguous()


def _flat(p):
    return p.reshape(-1)


class _RBFBase(nn.Module):
    input_dim = 2
    _batched = False        # True: parameters are per-factor, output keeps the leading L dimension
    _kind = 0               # covariance functor of the fused kernel build: 0 = RBF, 1 / 2 / 3 = Matern-3/2 / -1/2 / -5/2

    def _params(self):
        return _flat(self.sigma), _flat(self.lengthscale)

    def _group_coeff(self):
        return None

    def _build(self, X, Z, groupsX=None, groupsZ=None, jitter=0.0, want_lo=False, want_h=False):
        sigma, ls = self._params()
        dt = X.dtype
        sigma, ls = sigma.to(dt), ls.to(dt)
        if groupsX is not None:     # (a, r^2 table, groups of X, groups of Z, p_half)
            group = (self._group_coeff().to(dt), _r2_table(self.embedding, dt).to(X.device), groupsX, groupsZ,
                     0.5 * float(self.input_dim))
        else:
            group = (None, None, None, None, 1.0)
        if want_h:      # split-FP16 planes for the tensor-core predict: (stand-in for K, Kh, Kl, scale), leading L kept
            box = F.KernelBuildBox()       # lets the consumer of the planes launch this build's backward early (functional.py)
            out = F.KernelBuildH.apply(X, Z, sigma, ls, *group, float(jitter), self._kind, box)
            out[0]._gpz_box = box
            return out
        K = F.KernelBuild.apply(X, Z, sigma, ls, *group, float(jitter), want_lo, self._kind)
        if want_lo and isinstance(K, tuple):          # (K, K_lo): lo part for the split-TF32 tensor-core GEMMs
            return K if self._batched else (K[0][0], K[1][0])
        if want_lo:
            return K if self._batched else K[0], None
        return K if self._batched else K[0]

    def _diag(self, X):
        s2 = _flat(self.sigma) ** 2
        if self._batched:
            return s2[:, None].expand(-1, X.size(0))
        return s2.reshape(()).expand(X.size(0))

    def forward_distance(self, distance_squared):
        """sigma^2 exp(-0.5 d^2 / l^2) on a precomputed squared-distance tensor (kernels.py:128-130).
        Element-wise convenience kept for API compatibility; not on the fused hot path."""
        return (self.sigma ** 2) * torch.exp(-0.5 * distance_squared / (self.lengthscale ** 2))


class _MultiGroup:
    """forward of the multi-group kernels: points carry group labels (groupsX, groupsZ); diag=True is sigma^2, whatever the
    groups."""
    _input_dim_from_X = False       # True: p = X.shape[-1] on every call (batched_MGGP_RBF) instead of input_dim

    def forward(self, X, Z, groupsX, groupsZ, diag=False, _jitter=0.0, _want_lo=False, _want_h=False):
        if diag:
            return self._diag(X)
        if self._input_dim_from_X:
            self.input_dim = X.shape[-1]
        return self._build(X, Z, groupsX, groupsZ, jitter=_jitter, want_lo=_want_lo, want_h=_want_h)


class RBF(_RBFBase):
    def __init__(self, sigma=1.0, lengthscale=2.0):
        super().__init__()
        self.sigma = nn.Parameter(torch.tensor(sigma))
        self.lengthscale = nn.Parameter(torch.tensor(lengthscale))
        self.input_dim = 2

    def forward(self, X, Z, diag=False, return_distance=False, _jitter=0.0, _want_lo=False, _want_h=False):
        if diag:
            return self._diag(X)
        K = self._build(X, Z, jitter=_jitter, want_lo=_want_lo, want_h=_want_h)
        if return_distance:
            return K, F.cdist(X, Z)
        return K


class NSF_RBF(RBF):
    _batched = True

    def __init__(self, sigma=1.0, lengthscale=2.0, L=10):
        super().__init__(sigma=sigma, lengthscale=lengthscale)
        self.L = L
        self.sigma = nn.Parameter(sigma * torch.ones((L, 1, 1)))
        self.lengthscale = nn.Parameter(lengthscale * torch.ones((L, 1, 1)))


class MGGP_RBF(_MultiGroup, RBF):
    """Multi-group RBF, scalar parameters, coefficient a = group_diff_param (kernels.py:158-191)."""

    def __init__(self, sigma=1.0, lengthscale=2.0, group_diff_param=1.0, n_groups=2, device="cpu"):
        super().__init__(sigma, lengthscale)
        self.group_diff_param = nn.Parameter(torch.tensor(group_diff_param))
        self.embedding = embed_distance_matrix(torch.ones(n_groups, n_groups) - torch.eye(n_groups)).to(device)

    def set_group_distances(self, group_distances):
        self.embedding = embed_distance_matrix(group_distances)

    def _group_coeff(self):
        return _flat(self.group_diff_param)


class MGGP_NSF_RBF(_MultiGroup, NSF_RBF):
    """Per-factor multi-group RBF, a = group_diff_param**2 (kernels.py:194-228)."""

    def __init__(self, sigma=1.0, lengthscale=2.0, group_diff_param=1.0, n_groups=2, L=10, device="cpu"):
        super().__init__(sigma, lengthscale, L)
        self.group_diff_param = nn.Parameter(group_diff_param * torch.ones((L, 1, 1)))
        self.embedding = nn.Parameter(
            embed_distance_matrix(torch.ones(n_groups, n_groups) - torch.eye(n_groups)), requires_grad=False)

    def set_group_distances(self, group_distances):
        self.embedding = nn.Parameter(embed_distance_matrix(group_distances), requires_grad=False)

    def _group_coeff(self):
        return _flat(self.group_diff_param) ** 2


class batched_RBF(_RBFBase):
    """vmap-style RBF whose parameters may be scalars or (L,) vectors (kernels.py:32-59); same fused kernel.
    diag=True returns sigma^2 broadcast to (L, N) — the reference's expand at kernels.py:55 is shape-broken
    for 2-D X (SURVEY.md App. B) and is not reproduced."""

    def __init__(self, sigma=1.0, lengthscale=2.0):
        super().__init__()
        self.sigma = nn.Parameter(torch.as_tensor(sigma, dtype=torch.get_default_dtype()))
        self.lengthscale = nn.Parameter(torch.as_tensor(lengthscale, dtype=torch.get_default_dtype()))

    @property
    def _batched(self):
        return self.sigma.dim() > 0

    def _params(self):
        s, l = _flat(self.sigma), _flat(self.lengthscale)
        n = max(s.numel(), l.numel())
        return s.expand(n), l.expand(n)

    def forward(self, X, Z, diag=False, _jitter=0.0, _want_lo=False, _want_h=False):
        if diag:
            return self._diag(X)
        return self._build(X, Z, jitter=_jitter, want_lo=_want_lo, want_h=_want_h)


class batched_Matern32(batched_RBF):
    """Matern-3/2 covariance sigma^2 (1 + v) exp(-v), v = sqrt(3) |x - z| / lengthscale (kernels.py:6-30), scalar or (L,)
    parameters: the second covariance functor of the fused kernel build (`kind = 1` of gpz_kernel_build_*).  The analytic
    backward is finite at x == z, where the reference's autograd of sqrt(sum diff^2) returns NaN."""
    _kind = 1

    def forward_distance(self, distance_squared):
        v = (3.0 * distance_squared).sqrt() / self.lengthscale
        return (self.sigma ** 2) * (1 + v) * torch.exp(-v)


class batched_Matern12(batched_RBF):
    """Matern-1/2 (exponential) covariance sigma^2 exp(-v), v = |x - z| / lengthscale, scalar or (L,) parameters: `kind = 2`
    of gpz_kernel_build_*.  K has a cusp at x == z; the fused backward takes the sub-gradient 0 there (the position gradient
    of a coincident pair is exactly 0).  The reference has no counterpart of this class."""
    _kind = 2

    def forward_distance(self, distance_squared):
        return (self.sigma ** 2) * torch.exp(-distance_squared.sqrt() / self.lengthscale)


class batched_Matern52(batched_RBF):
    """Matern-5/2 covariance sigma^2 (1 + v + v^2/3) exp(-v), v = sqrt(5) |x - z| / lengthscale, scalar or (L,) parameters:
    `kind = 3` of gpz_kernel_build_*.  K is twice differentiable at x == z, and the fused backward is finite there (the position
    gradient of a coincident pair is exactly 0).  The reference has no counterpart of this class."""
    _kind = 3

    def forward_distance(self, distance_squared):
        v = (5.0 * distance_squared).sqrt() / self.lengthscale
        return (self.sigma ** 2) * (1 + v + v * v / 3) * torch.exp(-v)


class _ARDBase(_RBFBase):
    """Per-dimension (ARD) lengthscales: the covariance of `_kind` at unit lengthscale on the scaled squared distance
    s2 = sum_d (x_d - z_d)^2 / lengthscale[l, d]^2 (gpz_kernel_build_ard_*).  `sigma` is a scalar or (L,); `lengthscale` is
    (D,) or (L, D), its last axis always the input dimension (a scalar is broadcast to (dim,)).  Equal lengthscales along D
    give the isotropic kernel of the same kind.  There is no multi-group form, and VNNGP refuses these kernels."""
    _ard = True

    def __init__(self, sigma=1.0, lengthscale=2.0, dim=2):
        super().__init__()
        dt = torch.get_default_dtype()
        sigma = torch.as_tensor(sigma, dtype=dt)
        ls = torch.as_tensor(lengthscale, dtype=dt)
        if ls.dim() == 0:
            ls = ls.expand(dim).clone()
        if sigma.dim() > 1 or ls.dim() > 2:
            raise ValueError(f"{type(self).__name__}: sigma must be a scalar or (L,) and lengthscale (D,) or (L, D); got "
                             f"{tuple(sigma.shape)} and {tuple(ls.shape)}")
        self.sigma = nn.Parameter(sigma)
        self.lengthscale = nn.Parameter(ls)
        self._params()

    @property
    def input_dim(self):
        return self.lengthscale.shape[-1]

    @property
    def _batched(self):
        return self.sigma.dim() > 0 or self.lengthscale.dim() == 2

    def _params(self):
        """(sigma (L,), lengthscale (L, D))."""
        s, l = _flat(self.sigma), self.lengthscale
        Ls = s.numel() if self.sigma.dim() > 0 else None
        Ll = l.shape[0] if l.dim() == 2 else None
        if Ls is not None and Ll is not None and Ls != Ll:
            raise ValueError(f"{type(self).__name__}: sigma has L = {Ls} factors, lengthscale has L = {Ll}")
        L = Ls or Ll or 1
        return s.expand(L), l.reshape(-1, l.shape[-1]).expand(L, -1)

    def _diag(self, X):
        s2 = self._params()[0] ** 2
        return s2[:, None].expand(-1, X.size(0)) if self._batched else s2.reshape(()).expand(X.size(0))

    def forward(self, X, Z, diag=False, _jitter=0.0, _want_lo=False, _want_h=False):
        D = self.lengthscale.shape[-1]
        for name, t in (("X", X), ("Z", Z)):
            if t.dim() != 2 or t.shape[-1] != D:
                raise ValueError(f"{type(self).__name__}: {name} is {tuple(t.shape)}, expected (n, {D}) for its lengthscale's D")
        if diag:
            return self._diag(X)
        return self._build(X, Z, jitter=_jitter, want_lo=_want_lo, want_h=_want_h)

    def forward_distance(self, distance_squared):
        raise NotImplementedError(f"{type(self).__name__}: a summed squared distance has lost the per-dimension differences "
                                  "that per-dimension lengthscales scale")


class batched_ARD_RBF(_ARDBase):
    """RBF sigma^2 exp(-s2 / 2) with per-dimension lengthscales (`kind = 0` of gpz_kernel_build_ard_*)."""
    _kind = 0


class batched_ARD_Matern12(_ARDBase):
    """Matern-1/2 sigma^2 exp(-r), r = sqrt(s2), with per-dimension lengthscales (`kind = 2`); the backward takes the
    sub-gradient 0 at r = 0."""
    _kind = 2


class batched_ARD_Matern32(_ARDBase):
    """Matern-3/2 sigma^2 (1 + v) exp(-v), v = sqrt(3 s2), with per-dimension lengthscales (`kind = 1`)."""
    _kind = 1


class batched_ARD_Matern52(_ARDBase):
    """Matern-5/2 sigma^2 (1 + v + v^2/3) exp(-v), v = sqrt(5 s2), with per-dimension lengthscales (`kind = 3`)."""
    _kind = 3


class batched_MGGP_RBF(_MultiGroup, batched_RBF):
    """kernels.py:62-104: a = |group_diff_param|, p = X.shape[-1]."""
    _input_dim_from_X = True

    def __init__(self, sigma=1.0, lengthscale=1.0, group_diff_param=1.0, n_groups=10):
        super().__init__(sigma, lengthscale)
        self.group_diff_param = nn.Parameter(torch.as_tensor(group_diff_param, dtype=torch.get_default_dtype()))
        self.embedding = nn.Parameter(
            embed_distance_matrix(torch.ones(n_groups, n_groups) - torch.eye(n_groups)), requires_grad=False)

    def set_group_distances(self, group_distances):
        self.embedding = nn.Parameter(embed_distance_matrix(group_distances), requires_grad=False)

    def _group_coeff(self):
        n = self._params()[0].numel()
        return torch.abs(_flat(self.group_diff_param)).expand(n)
