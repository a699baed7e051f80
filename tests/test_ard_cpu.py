"""CPU: per-dimension (ARD) lengthscales: the five C entry points, the four kernel classes' parameters, their shape checks,
and VNNGP's refusal of them."""
import os

import pytest
import torch

import gpzoo_b200 as gz

CLASSES = (("batched_ARD_RBF", 0), ("batched_ARD_Matern12", 2), ("batched_ARD_Matern32", 1), ("batched_ARD_Matern52", 3))
ENTRY_POINTS = {"gpz_kernel_build_ard_fwd_f32": 13, "gpz_kernel_build_ard_fwd_f64": 13, "gpz_kernel_build_ard_fwd_h_f32": 14,
                "gpz_kernel_build_ard_bwd_f32": 16, "gpz_kernel_build_ard_bwd_f64": 16}


@pytest.fixture(scope="module")
def lib():
    from gpzoo_b200 import _cabi, build
    if not os.path.exists(_cabi.LIB_PATH):
        build.build()
    return _cabi.lib()


def test_entry_points_declared_exported_and_bound(lib):
    from gpzoo_b200 import _cabi
    protos = _cabi.prototypes()
    for sym, n in ENTRY_POINTS.items():
        assert sym in protos and sym in _cabi.exported_symbols(), sym
        assert len(protos[sym].params) == n, sym
        assert len(getattr(lib, sym).argtypes) == n, sym
        assert protos[sym].params[-1].name == "stream", sym
        names = [p.name for p in protos[sym].params]
        assert not {"a", "r2", "g1", "g2", "ng", "p_half"} & set(names), sym     # no group arguments
    assert lib.gpz_abi_version() == 4


@pytest.mark.parametrize("name,kind", CLASSES)
def test_kind_and_export(name, kind):
    cls = getattr(gz.kernels, name)
    assert cls._kind == kind and cls()._kind == kind and cls._ard


@pytest.mark.parametrize("name,kind", CLASSES)
def test_constructor_shapes_and_state_dict(name, kind):
    cls = getattr(gz.kernels, name)
    k = cls()                                                             # scalar lengthscale -> (dim,)
    assert k.lengthscale.shape == (2,) and k.sigma.shape == () and not k._batched
    assert list(k.state_dict()) == ["sigma", "lengthscale"]
    assert torch.equal(k.lengthscale.detach(), torch.full((2,), 2.0))
    assert cls(lengthscale=0.5, dim=3).lengthscale.shape == (3,)
    s, l = k._params()
    assert s.shape == (1,) and l.shape == (1, 2)

    k = cls(sigma=torch.ones(4), lengthscale=torch.tensor([1.0, 2.0, 3.0]))   # (L,) sigma, (D,) lengthscale shared by factors
    assert k._batched and k.input_dim == 3
    s, l = k._params()
    assert s.shape == (4,) and l.shape == (4, 3) and torch.equal(l[2], torch.tensor([1.0, 2.0, 3.0]))

    k = cls(sigma=1.5, lengthscale=torch.rand(5, 2) + 0.5)                    # scalar sigma, (L, D) lengthscale
    assert k._batched
    s, l = k._params()
    assert s.shape == (5,) and l.shape == (5, 2) and torch.equal(s, torch.full((5,), 1.5))
    assert k(torch.zeros(7, 2), torch.zeros(7, 2), diag=True).shape == (5, 7)
    assert torch.equal(k(torch.zeros(7, 2), torch.zeros(7, 2), diag=True), torch.full((5, 7), 1.5 ** 2))

    k = cls(sigma=torch.ones(3), lengthscale=torch.ones(3, 4))
    assert {n: tuple(p.shape) for n, p in k.state_dict().items()} == {"sigma": (3,), "lengthscale": (3, 4)}
    assert k(torch.zeros(6, 4), torch.zeros(6, 4), diag=True).shape == (3, 6)
    assert cls(sigma=1.1)(torch.zeros(6, 2), torch.zeros(6, 2), diag=True).shape == (6,)


@pytest.mark.parametrize("name,kind", CLASSES)
def test_mismatches_raise_value_error(name, kind):
    cls = getattr(gz.kernels, name)
    with pytest.raises(ValueError, match="L = 3"):
        cls(sigma=torch.ones(3), lengthscale=torch.ones(4, 2))
    with pytest.raises(ValueError):
        cls(lengthscale=torch.ones(2, 2, 2))
    k = cls(sigma=torch.ones(3), lengthscale=torch.ones(3, 2))
    X = torch.zeros(5, 3)                       # CPU tensors: a launch would raise GpzError, not ValueError
    with pytest.raises(ValueError, match="D|2"):
        k(X, X)
    with pytest.raises(ValueError):
        k(torch.zeros(5, 2), X)
    with pytest.raises(ValueError):
        k(X, X, diag=True)


@pytest.mark.parametrize("name,kind", CLASSES)
def test_forward_distance_raises(name, kind):
    with pytest.raises(NotImplementedError):
        getattr(gz.kernels, name)().forward_distance(torch.ones(3, 3))


@pytest.mark.parametrize("name,kind", CLASSES)
def test_vnngp_refuses_before_the_device(name, kind):
    v = gz.gp.VNNGP(getattr(gz.kernels, name)(), dim=2, M=8, K=3).double()
    X = torch.rand(16, 2, dtype=torch.float64)                # CPU tensors: any device call would raise GpzError instead
    with pytest.raises(NotImplementedError, match=name):
        v(X)


def test_functional_checks_ard_shape_and_groups():
    from gpzoo_b200 import _cabi, functional as F
    x = torch.zeros(4, 2, dtype=torch.float64)
    s = torch.ones(3, dtype=torch.float64)
    with pytest.raises(_cabi.GpzError, match="ARD"):
        F._check_kernel_args(x, x, s, torch.ones(3, 3, dtype=torch.float64), None, None, None, None)
    with pytest.raises(_cabi.GpzError, match="ARD"):
        F._check_kernel_args(x, x, s, torch.ones(2, 2, dtype=torch.float64), None, None, None, None)
    g = torch.zeros(4, dtype=torch.int64)
    with pytest.raises(_cabi.GpzError, match="multi-group"):
        F._check_kernel_args(x, x, s, torch.ones(3, 2, dtype=torch.float64), s, torch.zeros(2, 2, dtype=torch.float64), g, g)
