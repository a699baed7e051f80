"""GPU: the fp32 panel-hybrid Cholesky + inverse (`gpz_chol_inv_tc_f32`), whose work is split between the caller's stream and a
library-owned side stream: accuracy against float64, exact zeros above the diagonal, bit-identical repeats (the race detector for
the two-stream schedule), outputs that are final on the caller's stream, and the position of a failure in a late panel."""
import pytest
import torch

from tests.helpers import relerr

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 5e-5          # the fp32 tolerance of test_ops_gpu.py::test_cholesky_and_inverse


def _chol_inv(K):
    from gpzoo_b200 import functional as F
    assert K.dtype == torch.float32 and K.shape[-1] > F.CHOL_TC_MIN_M and K.shape[-1] % 4 == 0   # the hybrid path
    return F.CholeskyInverse.apply(K)


def _dense_spd(L, M, seed):
    g = torch.Generator().manual_seed(seed)
    Q = torch.randn(L, M, M, generator=g, dtype=torch.float64)
    return (Q @ Q.transpose(1, 2) / M + torch.eye(M, dtype=torch.float64)).to(DEV, torch.float32)


def _config2_kzz():
    import gpzoo_b200 as gz
    from gpzoo_b200 import synthetic
    pr = synthetic.nsf_problem(N=64, M=1024, L=10, G=4, E=1, seed=1, coord_scale=100.0, lengthscale=1.7, jitter=1e-1,
                               dtype=torch.float32, device=DEV)
    kern = gz.kernels.NSF_RBF(L=10)
    kern.sigma, kern.lengthscale = torch.nn.Parameter(pr["sigma"]), torch.nn.Parameter(pr["lengthscale"])
    with torch.no_grad():
        return kern(pr["Z"], pr["Z"], _jitter=pr["jitter"]).contiguous()


def _check(K):
    Lc, Linv = _chol_inv(K)
    ref = torch.linalg.cholesky(K.double())
    assert relerr(Lc, ref) < TOL
    assert relerr(Linv, torch.linalg.inv(ref)) < TOL
    assert torch.equal(Lc.triu(1), torch.zeros_like(Lc)) and torch.equal(Linv.triu(1), torch.zeros_like(Linv))
    return Lc, Linv


def test_config2_kzz_accuracy():
    _check(_config2_kzz())


@pytest.mark.parametrize("M", [1024, 1280, 1100])          # four panels, five panels, a ragged last panel
@pytest.mark.parametrize("L", [1, 10])
def test_dense_accuracy(M, L):
    _check(_dense_spd(L, M, seed=M + L))


def test_repeat_is_bit_identical():
    K = _dense_spd(10, 1280, seed=3)
    Lc0, Linv0 = _chol_inv(K)
    Lc1, Linv1 = _chol_inv(K)
    assert torch.equal(Lc0, Lc1) and torch.equal(Linv0, Linv1)
    Kc = _config2_kzz()
    a, b = _chol_inv(Kc), _chol_inv(Kc)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_bit_identical_with_work_queued_on_the_side_stream():
    from gpzoo_b200 import functional as F
    K = _dense_spd(10, 1024, seed=5)
    Lc0, Linv0 = _chol_inv(K)
    torch.cuda.synchronize()
    side = F.side_stream(torch.device(DEV))
    A = torch.randn(4096, 4096, device=DEV)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(40):                                     # unrelated work, long enough to overlap the whole call
            A = torch.tanh(A @ A * 1e-3)
    Lc1, Linv1 = _chol_inv(K)
    torch.cuda.current_stream().wait_stream(side)
    assert torch.equal(Lc0, Lc1) and torch.equal(Linv0, Linv1)


def test_outputs_final_on_the_callers_stream():
    K = _dense_spd(10, 1024, seed=6)
    Lc_ref, Linv_ref = _chol_inv(K)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):                                  # a stream the library has never seen
        Lc, Linv = _chol_inv(K)
        snap_lc, snap_linv = Lc.clone(), Linv.clone()           # read right after the call, no synchronisation
    torch.cuda.synchronize()
    assert torch.equal(snap_lc, Lc_ref) and torch.equal(snap_linv, Linv_ref)


def test_third_panel_failure_reports_first_bad_column():
    from gpzoo_b200 import functional as F
    K = _dense_spd(2, 1024, seed=7)
    K[1, 600, 600] = -5.0                                       # panel 2 (columns 512..767); leading minors up to 600 are fine
    W = K.clone()
    info = torch.full((2,), -1, dtype=torch.int32, device=DEV)
    Lc, Linv, tmp = torch.empty_like(W), torch.empty_like(W), torch.empty_like(W)
    lo_ws = torch.empty((4,) + tuple(W.shape), dtype=W.dtype, device=DEV)
    F.call("chol_inv_tc", W.dtype, W, Lc, Linv, tmp, lo_ws, 1024, 2, info)
    assert info.tolist() == [0, 601]
    with pytest.raises(torch.linalg.LinAlgError, match=r"Batch element 1\).*order 601"):
        _chol_inv(K)
