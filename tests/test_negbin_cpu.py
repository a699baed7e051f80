"""CPU: the negative-binomial likelihood's C ABI (gpz_negbin_*), the workspace size the library reports, and the NB model classes'
parameters and input checks."""
import math
import os

import pytest
import torch

from gpzoo_b200.counts import SparseCounts

from tests.test_poisson_shapes_gpu import SHAPES, _workspace_bytes, poisson_grid

NEW_SYMBOLS = ("gpz_negbin_workspace_bytes_f32", "gpz_negbin_workspace_bytes_f64", "gpz_negbin_fwdbwd_f32", "gpz_negbin_fwdbwd_f64",
               "gpz_negbin_fwdbwd_yt_f32", "gpz_digamma_f64", "gpz_lgamma_f64")


def _lib():
    from gpzoo_b200 import _cabi, build
    if not os.path.exists(_cabi.LIB_PATH):
        build.build()
    return _cabi.lib()


def _negbin_workspace_bytes(G, F, B, E, is_f32):
    """Mirror of negbin_ws_bytes in csrc/poisson.cu: the Poisson workspace, 16-byte aligned, then the d/dD partials [nbx][G]
    (16-byte aligned), the per-gene terms [G][2] and the tables [G][64][2]."""
    _, nbx, _, _ = poisson_grid(G, F, B, is_f32)
    elt = 4 if is_f32 else 8
    a16 = lambda n: -(-n // 16) * 16
    return a16(_workspace_bytes(G, F, B, E, is_f32)) + a16(elt * nbx * G) + elt * 130 * G


def test_header_exports_and_abi_version():
    from gpzoo_b200 import _cabi
    lib = _lib()
    assert lib.gpz_abi_version() == 4                      # entry points were only added
    syms = _cabi.exported_symbols()
    for s in NEW_SYMBOLS:
        assert s in syms, s
        assert hasattr(lib, s), s


def test_negbin_workspace_bytes_match_the_mirror():
    lib = _lib()
    for s in SHAPES.values():
        for F in (1, 10, 16, 17, 20, 32):
            for is_f32, suf in ((True, "f32"), (False, "f64")):
                args = (s["G"], F, s["B"] or s["Ntot"], s["E"])
                got = getattr(lib, "gpz_negbin_workspace_bytes_" + suf)(*args)
                assert got == _negbin_workspace_bytes(*args, is_f32), (args, suf)


def _models(y):
    import gpzoo_b200 as gz
    L = 3
    kern = gz.kernels.NSF_RBF(L=L)
    gp = gz.gp.SVGP(kern, dim=2, M=8)
    prior = gz.gp.GaussianPrior(y, L=2)
    return ((gz.likelihoods.NSF2, gz.likelihoods.NSF2_NB, (gp, y), dict(L=L)),
            (gz.likelihoods.PNMF, gz.likelihoods.PNMF_NB, (prior, y), dict(L=2)),
            (gz.likelihoods.Hybrid_NSF2, gz.likelihoods.Hybrid_NSF2_NB, (gp, prior, y), dict(L=L, T=2)))


def test_state_dict_is_the_parent_plus_dispersion():
    y = torch.poisson(torch.full((7, 30), 2.0))
    for parent, nb, args, kw in _models(y):
        p, m = parent(*args, **kw), nb(*args, **kw)
        assert isinstance(m, parent)
        keys_p, keys_m = set(p.state_dict()), set(m.state_dict())
        assert keys_m == keys_p | {"dispersion"}, (nb.__name__, keys_m ^ keys_p)
        assert tuple(m.dispersion.shape) == (7,)
        theta = torch.nn.functional.softplus(m.dispersion.detach().double())
        assert torch.allclose(theta, torch.ones(7, dtype=torch.float64), rtol=0, atol=1e-7)
        assert abs(float(m.dispersion[0]) - math.log(math.e - 1)) < 1e-7


def test_sparse_counts_raise_not_implemented():
    import gpzoo_b200 as gz
    y = torch.poisson(torch.full((7, 30), 2.0))
    ys = SparseCounts.from_dense(y)
    prior = gz.gp.GaussianPrior(y, L=2)
    m = gz.likelihoods.PNMF_NB(prior, ys, L=2)
    with pytest.raises(NotImplementedError, match="to_dense"):
        m.elbo(ys, E=1)


def test_cpu_tensors_raise_gpz_error():
    import gpzoo_b200 as gz
    from gpzoo_b200 import _cabi
    _lib()
    y = torch.poisson(torch.full((7, 30), 2.0))
    prior = gz.gp.GaussianPrior(y, L=2)
    m = gz.likelihoods.PNMF_NB(prior, y, L=2)
    with pytest.raises(_cabi.GpzError):
        m.elbo(y, E=1)
