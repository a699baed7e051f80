"""CPU: the sparse count format (gpzoo_b200.counts.SparseCounts) — conversions, canonical form, validation, spot slicing — and
the K7-CSC entry points of the C ABI."""
import os

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from gpzoo_b200.counts import SparseCounts


def _counts(G=13, N=21, density=0.3, seed=0, top=6):
    rng = np.random.default_rng(seed)
    y = rng.integers(1, top + 1, size=(G, N)) * (rng.random((G, N)) < density)
    y[:, 4] = 0                                          # an empty spot
    y[2, :] = 0                                          # an empty gene
    return torch.from_numpy(y.astype(np.float32))


def test_round_trips_scipy_csr_csc_and_dense():
    y = _counts()
    G, N = y.shape
    a = SparseCounts.from_scipy(sp.csr_matrix(y.numpy().T))                    # AnnData: N x G CSR
    b = SparseCounts.from_scipy(sp.csc_matrix(y.numpy()), genes_by_spots=True)  # G x N CSC
    c = SparseCounts.from_dense(y)
    for s in (a, b, c):
        assert s.shape == torch.Size((G, N)) and s.nnz == int((y != 0).sum())
        assert s.indptr.dtype == torch.int64 and s.genes.dtype == torch.int32 and s.values.dtype == torch.uint8
        assert torch.equal(s.to_dense(torch.float32), y)
        assert torch.equal(s.indptr, a.indptr) and torch.equal(s.genes, a.genes) and torch.equal(s.values, a.values)
    assert torch.equal(a.to_dense(torch.float64), y.double())
    # spot-major, genes ascending within a spot: the arrays of AnnData's CSR
    csr = sp.csr_matrix(y.numpy().T)
    assert np.array_equal(a.indptr.numpy(), csr.indptr) and np.array_equal(a.genes.numpy(), csr.indices)


def test_model_constructors_take_the_shape():
    import gpzoo_b200 as gz
    y = SparseCounts.from_dense(_counts())
    D, N = y.shape
    assert (D, N) == (13, 21)
    prior = gz.gp.GaussianPrior(y, L=2)
    assert tuple(prior.mean.shape) == (2, N)
    assert tuple(gz.likelihoods.PNMF(prior, y, L=2).V.shape) == (N,)


def test_duplicates_summed_and_zeros_dropped():
    # spot 0: gene 3 twice (1 + 2), an explicit zero at gene 1; spot 1: genes out of order
    rows = np.array([0, 0, 0, 1, 1])
    cols = np.array([3, 3, 1, 5, 2])
    data = np.array([1.0, 2.0, 0.0, 4.0, 7.0])
    m = sp.coo_matrix((data, (rows, cols)), shape=(3, 6))                     # N x G
    s = SparseCounts.from_scipy(m)
    assert s.indptr.tolist() == [0, 1, 3, 3]
    assert s.genes.tolist() == [3, 2, 5] and s.values.tolist() == [3, 7, 4]
    # the same from raw (unsorted, duplicated) arrays
    s2 = SparseCounts._build(torch.tensor([0, 3, 5, 5]), torch.tensor([3, 3, 1, 5, 2]), torch.tensor(data), 6, 3)
    assert torch.equal(s2.indptr, s.indptr) and torch.equal(s2.genes, s.genes) and torch.equal(s2.values, s.values)


@pytest.mark.parametrize("vals,dt", [([1, 255], torch.uint8), ([1, 256], torch.int16), ([3, 40000], torch.int32),
                                     ([1.5, 2.0], torch.float64), ([0.5, 1.0], torch.float32), ([1, 3 * 2 ** 31], torch.float64)])
def test_value_dtype(vals, dt):
    src = torch.tensor(vals, dtype=torch.float32 if dt == torch.float32 else torch.float64)
    s = SparseCounts._build(torch.tensor([0, 1, 2]), torch.tensor([0, 1]), src, 2, 2)
    assert s.values.dtype == dt
    assert torch.equal(s.values.double(), src.double())


def test_integer_input_dtype_kept_exact():
    m = sp.csr_matrix(np.array([[0, 70000], [5, 0]], dtype=np.int64))
    s = SparseCounts.from_scipy(m)
    assert s.values.dtype == torch.int32 and s.values.tolist() == [70000, 5]


def test_validation_errors():
    ip, g, v = torch.tensor([0, 2, 3]), torch.tensor([0, 1, 1]), torch.tensor([1.0, 2.0, 3.0])
    SparseCounts._build(ip, g, v, 2, 2)
    with pytest.raises(ValueError):
        SparseCounts._build(ip, torch.tensor([0, 2, 1]), v, 2, 2)          # gene out of range
    with pytest.raises(ValueError):
        SparseCounts._build(ip, torch.tensor([0, -1, 1]), v, 2, 2)
    with pytest.raises(ValueError):
        SparseCounts._build(torch.tensor([0, 3, 2]), g, v, 2, 2)           # not monotone
    with pytest.raises(ValueError):
        SparseCounts._build(torch.tensor([0, 1, 2]), g, v, 2, 2)           # does not end at nnz
    with pytest.raises(ValueError):
        SparseCounts._build(torch.tensor([0, 3]), g, v, 2, 2)              # wrong length
    with pytest.raises(ValueError):
        SparseCounts._build(ip, g, torch.tensor([1.0, -2.0, 3.0]), 2, 2)   # negative
    with pytest.raises(ValueError):
        SparseCounts._build(ip, g, torch.tensor([1.0, float("nan"), 3.0]), 2, 2)
    with pytest.raises(ValueError):
        SparseCounts.from_dense(-_counts())
    with pytest.raises(TypeError):
        SparseCounts.from_scipy(np.ones((2, 2)))


def test_spot_slices_and_other_indexing():
    y = _counts(N=40)
    s = SparseCounts.from_dense(y)
    for lo, hi in ((0, 40), (3, 17), (4, 5), (39, 40), (10, 10), (-5, None), (None, 7)):
        part = s[:, lo:hi]
        assert torch.equal(part.to_dense(), y[:, lo:hi]), (lo, hi)
        assert int(part.indptr[0]) == 0 and part.shape == y[:, lo:hi].shape
    for bad in (0, (slice(None), 3), (slice(None), slice(0, 10, 2)), (slice(0, 3), slice(0, 4)), slice(0, 4),
                (slice(None), torch.tensor([1, 2]))):
        with pytest.raises(TypeError):
            s[bad]


@pytest.mark.parametrize("world", [1, 3, 4])
def test_shards_concatenate_to_the_whole(world):
    from gpzoo_b200 import distributed
    y = _counts(N=37, seed=world)
    s = SparseCounts.from_dense(y)
    parts = [s[:, slice(*distributed.shard_range(37, world, r))] for r in range(world)]
    assert sum(p.nnz for p in parts) == s.nnz
    assert torch.equal(torch.cat([p.to_dense() for p in parts], 1), y)
    assert torch.equal(torch.cat([p.genes for p in parts]), s.genes)


def test_to_and_pin_memory_on_cpu():
    s = SparseCounts.from_dense(_counts())
    t = s.to("cpu")
    assert t.device.type == "cpu" and torch.equal(t.to_dense(), s.to_dense())
    assert s.dtype == torch.uint8 and "nnz" in repr(s)


def test_package_exports_and_abi():
    import gpzoo_b200 as gz
    from gpzoo_b200 import _cabi, build
    assert gz.SparseCounts is SparseCounts
    if not os.path.exists(_cabi.LIB_PATH):
        build.build()
    lib = _cabi.lib()
    assert lib.gpz_abi_version() == 4
    syms = _cabi.exported_symbols()
    for s in ("gpz_poisson_csc_workspace_bytes_f32", "gpz_poisson_csc_workspace_bytes_f64", "gpz_poisson_fwdbwd_csc_f32",
              "gpz_poisson_fwdbwd_csc_f64"):
        assert s in syms and hasattr(lib, s), s
    # large G: the G x F double accumulator of the atomic path is part of the (int64) workspace size
    assert lib.gpz_poisson_csc_workspace_bytes_f32(40000, 32, 10 ** 6, 1) > 8 * 40000 * 32


def test_sparse_counts_refused_on_cpu():
    """The kernel call refuses CPU arrays like every other entry point (there is no host path)."""
    import gpzoo_b200 as gz
    from gpzoo_b200 import _cabi, build
    if not os.path.exists(_cabi.LIB_PATH):
        build.build()
    y = SparseCounts.from_dense(_counts())
    G, N = y.shape
    W, V = torch.rand(G, 3), torch.zeros(N)
    mean, spread, eps = torch.zeros(3, N), torch.ones(3, N), torch.zeros(1, 3, N)
    with pytest.raises(_cabi.GpzError):
        gz.functional.PoissonLL.apply(y, None, W, V, mean, spread, eps, 0, 0.0, True, True)
