"""Sparse count matrices for the fused Poisson ELBO.

`SparseCounts` holds a G x N (genes x spots) count matrix as spot-major compressed columns — the same arrays as AnnData's
N x G CSR `adata.X`:

    indptr  int64, N + 1      spot n owns entries indptr[n] .. indptr[n + 1]
    genes   int32, nnz        gene of each entry, ascending within a spot
    values  nnz               uint8 / int16 / int32 for integral counts (the narrowest that holds them), else float32 / float64

Every model's `elbo` accepts it wherever it accepts a dense `y`; the likelihood kernel then reads only the nonzeros
(`functional.PoissonLL`, csrc/poisson.cu K7-CSC).  Entries are canonical — duplicates summed, explicit zeros dropped, genes
sorted — and validated once, when the object is built; nothing is checked per step beyond shapes.
"""
from __future__ import annotations

import torch

_INT_KINDS = ((torch.uint8, 255), (torch.int16, 32767), (torch.int32, 2 ** 31 - 1))


class SparseCounts:
    """G x N count matrix in spot-major compressed columns (see the module docstring).  Build it with `from_scipy` or
    `from_dense`; `y[:, lo:hi]` is a contiguous block of spots."""

    __slots__ = ("indptr", "genes", "values", "n_genes")

    def __init__(self, indptr, genes, values, n_genes):
        """Internal: wraps arrays that are already canonical.  Use `from_scipy` / `from_dense`."""
        self.indptr, self.genes, self.values, self.n_genes = indptr, genes, values, int(n_genes)

    # ---- construction ----------------------------------------------------------------------------------------------------
    @classmethod
    def from_scipy(cls, m, genes_by_spots=False):
        """From a scipy sparse matrix: N x G (spots x genes, AnnData's `adata.X`) by default, G x N with genes_by_spots=True.
        Any scipy format; the input is not modified."""
        import scipy.sparse as sp
        if not sp.issparse(m):
            raise TypeError(f"expected a scipy sparse matrix, got {type(m).__name__}")
        csr = sp.csr_matrix(m.T if genes_by_spots else m)          # rows = spots, columns = genes
        N, G = csr.shape
        return cls._build(torch.from_numpy(csr.indptr.astype("int64")), torch.from_numpy(csr.indices.astype("int64")),
                          torch.from_numpy(csr.data.copy()), G, N)

    @classmethod
    def from_dense(cls, y):
        """From a dense G x N tensor (any device, any real dtype); the result lives on the same device."""
        y = torch.as_tensor(y)
        if y.dim() != 2:
            raise ValueError(f"expected a G x N matrix, got shape {tuple(y.shape)}")
        G, N = y.shape
        yt = y.t()                                                   # N x G: nonzero() enumerates spot-major, genes ascending
        nz = yt.nonzero()
        spot, gene = nz[:, 0], nz[:, 1]
        indptr = torch.zeros(N + 1, dtype=torch.int64, device=y.device)
        indptr[1:] = torch.cumsum(torch.bincount(spot, minlength=N), 0)
        return cls._build(indptr, gene, yt[spot, gene], G, N)

    @classmethod
    def _build(cls, indptr, genes, values, G, N):
        """Validate, canonicalise (sort genes within a spot, sum duplicates, drop zeros) and pick the value dtype."""
        if values.dtype == torch.bool or values.is_complex():
            raise ValueError(f"counts must be real numbers, got {values.dtype}")
        indptr, genes = indptr.to(torch.int64), genes.to(torch.int64)
        nnz = genes.numel()
        if indptr.dim() != 1 or indptr.numel() != N + 1 or values.numel() != nnz:
            raise ValueError(f"indptr must have N + 1 = {N + 1} entries and values one per gene index")
        if int(indptr[0]) != 0 or int(indptr[-1]) != nnz or bool((indptr[1:] < indptr[:-1]).any()):
            raise ValueError("indptr must start at 0, be non-decreasing and end at nnz")
        if nnz and (int(genes.min()) < 0 or int(genes.max()) >= G):
            raise ValueError(f"gene index out of range [0, {G})")
        if nnz and not bool(((values >= 0) & torch.isfinite(values)).all()):
            raise ValueError("counts must be finite and non-negative")
        exact = not values.is_floating_point()
        acc = values.to(torch.int64 if exact else torch.float64)
        spot = torch.repeat_interleave(torch.arange(N, device=indptr.device), indptr[1:] - indptr[:-1])
        key = spot * G + genes
        if nnz > 1 and not bool((key[1:] > key[:-1]).all()):       # unsorted or duplicated entries
            key, order = torch.sort(key, stable=True)
            key, inv = torch.unique_consecutive(key, return_inverse=True)
            acc = torch.zeros(key.numel(), dtype=acc.dtype, device=acc.device).index_add_(0, inv, acc[order])
        keep = acc != 0
        key, acc = key[keep], acc[keep]
        spot, genes = key // G, key % G
        indptr = torch.zeros(N + 1, dtype=torch.int64, device=key.device)
        indptr[1:] = torch.cumsum(torch.bincount(spot, minlength=N), 0)
        return cls(indptr, genes.to(torch.int32), _narrow(acc, values.dtype), G)

    # ---- properties ------------------------------------------------------------------------------------------------------
    @property
    def shape(self):
        return torch.Size((self.n_genes, self.indptr.numel() - 1))

    @property
    def nnz(self):
        return self.genes.numel()

    @property
    def device(self):
        return self.genes.device

    @property
    def dtype(self):
        """dtype of the stored values."""
        return self.values.dtype

    def __repr__(self):
        G, N = self.shape
        return f"SparseCounts(shape=({G}, {N}), nnz={self.nnz}, values={self.values.dtype}, device={self.device})"

    # ---- movement --------------------------------------------------------------------------------------------------------
    def to(self, device, non_blocking=False):
        return SparseCounts(*(t.to(device, non_blocking=non_blocking) for t in (self.indptr, self.genes, self.values)), self.n_genes)

    def cuda(self, device=None, non_blocking=False):
        return self.to(torch.device("cuda") if device is None else device, non_blocking=non_blocking)

    def cpu(self):
        return self.to("cpu")

    def pin_memory(self):
        return SparseCounts(self.indptr.pin_memory(), self.genes.pin_memory(), self.values.pin_memory(), self.n_genes)

    def to_dense(self, dtype=torch.float32):
        """The G x N dense matrix, on the same device."""
        G, N = self.shape
        out = torch.zeros(G, N, dtype=dtype, device=self.device)
        spot = torch.repeat_interleave(torch.arange(N, device=self.device), self.indptr[1:] - self.indptr[:-1])
        out[self.genes.long(), spot] = self.values.to(dtype)
        return out

    # ---- slicing ---------------------------------------------------------------------------------------------------------
    def __getitem__(self, key):
        """y[:, lo:hi] — the contiguous block of spots lo .. hi - 1 (indptr rebased).  Any other index raises TypeError."""
        if not (isinstance(key, tuple) and len(key) == 2 and key[0] == slice(None) and isinstance(key[1], slice)
                and key[1].step in (None, 1)):
            raise TypeError("SparseCounts supports only y[:, lo:hi] (a contiguous block of spots)")
        lo, hi, _ = key[1].indices(self.shape[1])
        hi = max(lo, hi)
        ip = self.indptr[lo:hi + 1]
        a, b = int(ip[0]), int(ip[-1])
        return SparseCounts(ip - a, self.genes[a:b], self.values[a:b], self.n_genes)


def _narrow(v, src_dtype):
    """uint8 / int16 / int32 when every value is an integer count that fits, else float32 (float32 input) / float64."""
    if v.numel() == 0 or not v.is_floating_point() or bool((v == torch.round(v)).all()):
        top = int(v.max()) if v.numel() else 0
        for dt, lim in _INT_KINDS:
            if top <= lim:
                return v.to(dt)
    return v.to(torch.float32 if src_dtype in (torch.float32, torch.float16, torch.bfloat16) else torch.float64)
