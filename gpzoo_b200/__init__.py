"""gpzoo_b200 — B200-native (sm_100a) implementation of GPzoo's sparse-GP ELBO hot path.

Drop-in for `gpzoo.kernels`, `gpzoo.gp`, `gpzoo.likelihoods` (+ the hot-path part of `gpzoo.utilities`):

    import gpzoo_b200 as gpzoo          # or gpzoo_b200.install_as_gpzoo(); import gpzoo.kernels ...

All arithmetic runs in hand-written CUDA kernels reached through the C ABI in include/gpzoo_b200.h
(`gpzoo_b200/lib/libgpzoo_b200.so`); there is no CPU or PyTorch fallback — operations raise if the library
is missing or the tensors are not on a CUDA device.
"""
import sys as _sys

from . import _cabi, counts, functional, gp, kernels, likelihoods, optim, synthetic, utilities  # noqa: F401
from .counts import SparseCounts

__all__ = ["kernels", "gp", "likelihoods", "utilities", "optim", "functional", "synthetic", "counts", "SparseCounts",
           "install_as_gpzoo"]


def install_as_gpzoo():
    """Register this package under the reference's import path (`gpzoo`, `gpzoo.kernels`, ...)."""
    me = _sys.modules[__name__]
    _sys.modules["gpzoo"] = me
    for sub in ("kernels", "gp", "likelihoods", "utilities"):
        _sys.modules["gpzoo." + sub] = getattr(me, sub)
    return me
