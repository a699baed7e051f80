"""CPU: the Matern-1/2 and Matern-5/2 kernel classes (kinds 2 and 3 of the fused kernel build): exports, parameters,
the element-wise `forward_distance` against the closed forms, and VNNGP's refusal of them."""
import math
import sys

import pytest
import torch

import gpzoo_b200 as gz

NEW = (("batched_Matern12", 2), ("batched_Matern52", 3))


def _closed_form(kind, s, l, d2):
    r = math.sqrt(d2)
    if kind == 2:
        return s * s * math.exp(-r / l)
    v = math.sqrt(5.0) * r / l
    return s * s * (1.0 + v + v * v / 3.0) * math.exp(-v)


@pytest.mark.parametrize("name,kind", NEW)
def test_exported_with_kind(name, kind):
    cls = getattr(gz.kernels, name)
    assert cls._kind == kind and cls()._kind == kind
    assert issubclass(cls, gz.kernels.batched_RBF)
    saved = {k: v for k, v in sys.modules.items() if k == "gpzoo" or k.startswith("gpzoo.")}
    try:
        gz.install_as_gpzoo()
        import gpzoo.kernels
        assert getattr(gpzoo.kernels, name) is cls
    finally:
        for k in [k for k in sys.modules if k == "gpzoo" or k.startswith("gpzoo.")]:
            del sys.modules[k]
        sys.modules.update(saved)


@pytest.mark.parametrize("name,kind", NEW)
@pytest.mark.parametrize("params", [dict(sigma=1.3, lengthscale=0.7),
                                    dict(sigma=torch.linspace(1.0, 2.0, 4), lengthscale=torch.linspace(0.5, 1.5, 4))])
def test_state_dict_matches_matern32(name, kind, params):
    ours = getattr(gz.kernels, name)(**params).state_dict()
    ref = gz.kernels.batched_Matern32(**params).state_dict()
    assert list(ours) == list(ref)
    for k in ref:
        assert ours[k].shape == ref[k].shape and ours[k].dtype == ref[k].dtype, k
        assert torch.equal(ours[k], ref[k]), k


@pytest.mark.parametrize("name,kind", NEW)
def test_forward_distance_closed_form(name, kind):
    g = torch.Generator().manual_seed(3)
    d2 = 4.0 * torch.rand(5, 7, generator=g, dtype=torch.float64)
    d2[0, 0] = 0.0
    d2[1, 2] = 1e-30
    # scalar parameters
    k = getattr(gz.kernels, name)(sigma=1.3, lengthscale=0.7).double()
    k.sigma.data, k.lengthscale.data = torch.tensor(1.3, dtype=torch.float64), torch.tensor(0.7, dtype=torch.float64)   # (ctor: fp32)
    out = k.forward_distance(d2)
    ref = torch.tensor([[_closed_form(kind, 1.3, 0.7, float(x)) for x in row] for row in d2], dtype=torch.float64)
    assert out.dtype == torch.float64 and out.shape == d2.shape
    assert torch.allclose(out, ref, rtol=1e-14, atol=0)
    assert float(out[0, 0].detach()) == pytest.approx(1.3 ** 2, rel=1e-15)
    # (L,) parameters against an (L, n, m) squared-distance tensor
    L = 3
    sg = torch.tensor([0.9, 1.1, 1.6], dtype=torch.float64)
    ls = torch.tensor([0.4, 1.0, 2.5], dtype=torch.float64)
    kb = getattr(gz.kernels, name)(sigma=sg, lengthscale=ls).double()
    kb.sigma.data, kb.lengthscale.data = sg.reshape(L, 1, 1).clone(), ls.reshape(L, 1, 1).clone()
    outb = kb.forward_distance(d2.expand(L, -1, -1))
    refb = torch.tensor([[[_closed_form(kind, float(sg[l]), float(ls[l]), float(x)) for x in row] for row in d2] for l in range(L)],
                        dtype=torch.float64)
    assert torch.allclose(outb, refb, rtol=1e-14, atol=0)


@pytest.mark.parametrize("name,kind", NEW)
def test_vnngp_refuses_before_the_device(name, kind):
    v = gz.gp.VNNGP(getattr(gz.kernels, name)(), dim=2, M=8, K=3).double()
    X = torch.rand(16, 2, dtype=torch.float64)                # CPU tensors: any device call would raise GpzError instead
    with pytest.raises(NotImplementedError, match=name):
        v(X)
