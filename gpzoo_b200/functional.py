"""torch.autograd.Functions over the C ABI (include/gpzoo_b200.h).

The reference gets every gradient from autograd over stock ATen ops (utilities.py:485,620
`loss.backward()`); here each fused CUDA kernel has a hand-written backward kernel and these Functions
only allocate tensors and pass pointers.  Maths: SURVEY.md Appendix A (validated against the reference).
All Functions work on L-batched, contiguous CUDA tensors in float32 or float64.
"""
from __future__ import annotations

import os
import sys

import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from . import _cabi
from ._cabi import call
from .counts import SparseCounts

# When True (default) a non-positive-definite Kzz raises torch.linalg.LinAlgError right away like the
# reference's torch.linalg.cholesky (one device sync).  Throughput runs may turn it off and call
# `check_cholesky_info()` when they read the loss.
SYNC_CHECKS = True
USE_TENSOR_CORES = True      # fp32: route large contractions through the tcgen05 kernels
# arithmetic of the N-proportional tensor-core GEMMs (K3/K4 and backward): "fp16x3" = split-FP16 (fp16 operand planes, f16 MMA
# rate), "tf32x3" = split-TF32 (fp32 + lo planes, half the rate; also used when a shape is not 8-aligned)
TENSOR_CORE_ARITH = os.environ.get("GPZ_TC_ARITH", "fp16x3")
# fp32 models: up to this many inducing points the O(M^3) chain runs in fp64 (gp.py `_chain_dtype`); GPZ_CHAIN_FP64_MAX_M=0 turns it off
CHAIN_FP64_MAX_M = int(os.environ.get("GPZ_CHAIN_FP64_MAX_M", "256"))
FUSED_CHAIN = os.environ.get("GPZ_FUSED_CHAIN", "1") != "0"
# chain + predict as one autograd node with the merged backward (SvgpMomentsH); GPZ_FUSED_MOMENTS=0: the two-node path
FUSED_MOMENTS = os.environ.get("GPZ_FUSED_MOMENTS", "1") != "0"       # csrc/chain.cu instead of the Function-per-op chain
CHOL_TC_MIN_M = int(os.environ.get("GPZ_CHOL_TC_MIN_M", "768"))   # above this size the fp32 Cholesky + inverse is the panel hybrid:
# 256-wide diagonal blocks on the cluster kernel, trailing updates and the inverse's doubling on tcgen05 (measured, L = 10:
# M = 512 0.42 vs 0.51 ms, M = 1024 1.30 vs 1.18 ms, M = 1536 3.41 vs 2.02 ms, cluster vs hybrid)
_pending_info = []
# build Kzx on a side stream, concurrently with the Cholesky chain of Kzz (gp.py moments); GPZ_OVERLAP=0 turns it off
OVERLAP_KERNEL_BUILD = os.environ.get("GPZ_OVERLAP", "1") != "0"
_side_streams = {}
launch_on = _cabi.launch_on


def side_stream(device):
    """The per-device side stream used for work that is independent of the Kzz chain."""
    key = torch.device(device).index if torch.device(device).index is not None else torch.cuda.current_device()
    st = _side_streams.get(key)
    if st is None:
        st = _side_streams[key] = torch.cuda.Stream(device=key)
        # the kernel-build backward runs on this stream by design; autograd orders it against the parameters' accumulation on the
        # main stream (that synchronisation is wanted) and would otherwise print a one-off warning about the stream mismatch
        mute = getattr(torch.autograd.graph, "set_warn_on_accumulate_grad_stream_mismatch", None)
        if mute is not None and os.environ.get("GPZ_NO_MUTE") != "1":
            mute(False)
    return st


def set_sync_checks(flag: bool):
    global SYNC_CHECKS
    SYNC_CHECKS = bool(flag)


_pending_amax = {}        # (names, device) -> running max of amax * scale of the split-FP16 predict calls not examined yet


def check_cholesky_info():
    """Deferred error checks of the step (one device sync): LAPACK-style `info` of every Cholesky and the overflow guard of
    the split-FP16 planes (a scale bound that did not hold makes an entry inf, which shows up as a non-finite tracked max)."""
    global _pending_info, _pending_amax
    pend16, _pending_amax = _pending_amax, {}
    pend, _pending_info = _pending_info, []          # both are cleared before anything can raise
    for (names, _dev), v in pend16.items():
        bad = ~(v <= 65504.0)                          # also true for NaN / inf
        if bool(bad.any()):
            which = sorted({names[int(i)] for i in bad.nonzero()[:, 0]})
            raise _cabi.GpzError("split-FP16 predict: " + ", ".join(which) + " left the fp16 range its scale bound allows (or the "
                                 "inputs contain inf/NaN); GPZ_TC_ARITH=tf32x3 selects the split-TF32 kernels")
    for info in pend:
        bad = info.nonzero()
        if bad.numel():
            l = int(bad[0, 0])
            raise torch.linalg.LinAlgError(
                f"gpzoo_b200.cholesky: (Batch element {l}): the input is not positive-definite "
                f"(leading minor of order {int(info[l])} is not positive-definite)")


def _track_info(info):
    """Queue a Cholesky `info` vector for the deferred check; long unsynchronised runs fold the queue (largest non-zero minor
    per factor, one launch per distinct shape) so that it stays bounded and no failure is dropped."""
    global _pending_info
    _pending_info.append(info)
    if len(_pending_info) > 256:
        groups = {}
        for t in _pending_info:
            groups.setdefault((tuple(t.shape), t.device), []).append(t)
        _pending_info = [torch.stack(g).amax(dim=0) for g in groups.values()]


def _track_amax(amax, scale, names):
    """Queue the overflow guard of one split-FP16 call: a running maximum of amax * scale per name on the device (two small
    launches, no sync, nothing retained from the call; torch.maximum propagates NaN).  Examined by check_cholesky_info()."""
    v = amax * scale
    key = (names, v.device)
    cur = _pending_amax.get(key)
    if cur is None or cur.shape != v.shape:
        if cur is not None:
            v = torch.maximum(v, cur.amax(dim=-1, keepdim=True).expand_as(v))
        _pending_amax[key] = v
    else:
        torch.maximum(cur, v, out=cur)


def _c(t):
    return t if t.is_contiguous() else t.contiguous()


# Scratch that lives only inside one backward call (the A diag(2 gv) and dL/dA planes: 2 x 4 L M N bytes, the chain backward's
# M x M workspaces) is kept resident per (purpose, device, stream) instead of going through the caching allocator every step:
# requests of 0.67 GB and 1.34 GB interleaved made the allocator split and re-grow its pool for dozens of steps (a cudaMalloc of
# 1.3 GB inside a backward stalls the host for ~100 ms; bench.py round 2 saw 8.5 -> 19 ms/step from it).  Reuse is safe because a
# buffer is written and consumed by launches of ONE Function.backward call on ONE stream, and the next use is ordered behind
# them on that stream.  `release_workspaces()` returns the memory.
_workspaces = {}
_workspace_readers = {}     # (purpose, stream) -> event of the last launch on ANOTHER stream that read the workspace


def _workspace(tag, shape, dtype, device):
    device = torch.device(device)
    idx = device.index if device.index is not None else torch.cuda.current_device()
    key = (tag, idx, torch.cuda.current_stream(idx).cuda_stream)
    n = 1
    for d in shape:
        n *= int(d)
    nbytes = n * torch.empty((), dtype=dtype).element_size()
    buf = _workspaces.get(key)
    if buf is None or buf.numel() < nbytes:
        _workspaces.pop(key, None)
        buf = _workspaces[key] = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=device)
    return buf[:nbytes].view(dtype).view(*shape)


def release_workspaces():
    """Drop the resident backward scratch (it is re-created on the next step)."""
    _workspaces.clear()
    _workspace_readers.clear()


def _plane_pair(L, m, n, device):
    """(hi, lo) fp16 planes as ONE allocation of 4 L m n bytes -- the size of every other large tensor of the step (fp32 dL/dKzx,
    the other plane pairs), so that the caching allocator reuses blocks one-to-one and never splits them."""
    pair = torch.empty((2, L, m, n), dtype=torch.float16, device=device)
    return pair[0], pair[1]


def gemm(A, B, ta=False, tb=False, alpha=1.0, beta=0.0, out=None, a_tri=0, b_tri=0, d_tri=0, splitk=1):
    """out[b] = alpha op(A[b]) op(B[b]) + beta out[b]; A, B, out are (batch, rows, cols) contiguous.

    fp32 products with all dimensions >= 128 go to the tcgen05 split-TF32 kernel (the M x M operand is split into
    (x, lo) / transposed on the fly); everything else, and all of fp64, runs on the exact CUDA-core GEMM."""
    bsz = A.shape[0]
    m, k = (A.shape[2], A.shape[1]) if ta else (A.shape[1], A.shape[2])
    n = B.shape[1] if tb else B.shape[2]
    kb = B.shape[2] if tb else B.shape[1]
    assert kb == k and B.shape[0] == bsz, (A.shape, B.shape, ta, tb)
    if out is None:
        out = (torch.zeros if (d_tri or splitk > 1) else torch.empty)((bsz, m, n), dtype=A.dtype, device=A.device)
    dt = A.dtype
    if (USE_TENSOR_CORES and TENSOR_CORE_ARITH == "fp16x3" and dt == torch.float32 and min(m, n, k) >= GEMM16_MIN_DIM
            and splitk == 1 and beta in (0.0, 1.0) and m % 8 == 0 and n % 8 == 0 and k % 8 == 0):
        # large products: split-FP16 (twice the tensor-core rate; the two operand passes are O(M^2) and only pay off here)
        Ah, Al, sa = split16_cached(A, transposed=ta)
        Bh, Bl, sb = split16_cached(B)
        umma_gemm16((Ah, Al, sa), (Bh, Bl, sb), int(tb), a_tri=a_tri, b_tri=b_tri, d_tri=d_tri, alpha=alpha,
                    Cin=out if beta == 1.0 else None, out=out)
        return out
    if (USE_TENSOR_CORES and dt == torch.float32 and min(m, n, k) >= 128 and splitk == 1 and beta in (0.0, 1.0)
            and m % 4 == 0 and n % 4 == 0 and k % 4 == 0):
        if ta:
            Ae, Ae_lo = transpose_lo(A)
        else:
            Ae, Ae_lo = A, tf32_lo(A)
        call("umma_gemm", dt, int(tb), m, n, k, alpha, Ae, Ae_lo, k, m * k, B, tf32_lo(B), B.shape[2], B.shape[1] * B.shape[2],
             out if beta == 1.0 else None, out, None, n, m * n, bsz, a_tri, b_tri, d_tri, 1, 3)
        return out
    call("gemm", dt, int(ta), int(tb), m, n, k, alpha,
         A, A.shape[2], A.shape[1] * A.shape[2],
         B, B.shape[2], B.shape[1] * B.shape[2],
         beta, out, out.shape[2], out.shape[1] * out.shape[2],
         bsz, a_tri, b_tri, d_tri, splitk)
    return out


GEMM16_MIN_DIM = 2048        # M x M x M products at least this large go to the split-FP16 kernel


def split16_cached(x, transposed=False):
    """(h, l, scale) fp16 planes of x — or, transposed=True, of its per-matrix transpose — cached for the duration of a step
    (the pass that writes the transposed planes writes the plain ones too and fills both cache entries)."""
    x = _c(x)
    if not transposed:
        hit = _step_cache.get(("h16T", x.data_ptr(), x._version, tuple(x.shape)))
        if hit is not None:
            h, l, _, _, sc = hit[0]
            return h, l, sc
        return _cached("h16", x, lambda: split16(x))
    h, l, hT, lT, sc = _cached("h16T", x, lambda: split16(x, transpose=True))
    return hT, lT, sc


def transpose_lo(x):
    """(x^T, lo(x^T)) per matrix of a batch of square fp32 matrices."""
    x = _c(x)

    def make():
        xt, xt_lo = torch.empty_like(x), torch.empty_like(x)
        call("transpose_lo", torch.float32, x, xt, xt_lo, x.shape[-1], x.shape[0])
        return xt, xt_lo
    return _cached("T", x, make)


class BatchedMatmul(Function):
    """A @ B for (batch, m, k) x (batch, k, n) through `gemm` (C-ABI GEMMs), with gA = g B^T and gB = A^T g."""

    @staticmethod
    def forward(ctx, A, B):
        A, B = _c(A), _c(B)
        ctx.save_for_backward(A, B)
        return gemm(A, B)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        A, B = ctx.saved_tensors
        g = _c(g)
        return (gemm(g, B, tb=True) if ctx.needs_input_grad[0] else None,
                gemm(A, g, ta=True) if ctx.needs_input_grad[1] else None)


def matmul(A, B):
    """Batched matrix product on the library's GEMM kernels; 2-D operands are treated as a batch of one and a 2-D / 3-D mix
    broadcasts the 2-D operand over the batch."""
    a3, b3 = A.dim() == 3, B.dim() == 3
    A3 = A if a3 else A.unsqueeze(0)
    B3 = B if b3 else B.unsqueeze(0)
    nb = max(A3.shape[0], B3.shape[0])
    if A3.shape[0] != nb:
        A3 = A3.expand(nb, -1, -1)
    if B3.shape[0] != nb:
        B3 = B3.expand(nb, -1, -1)
    out = BatchedMatmul.apply(A3, B3)
    return out if (a3 or b3) else out[0]


class SquaredDist(Function):
    """|x_i - z_j|^2 by direct differences (the `cdist` kernel squared), with the gradients to both point sets."""

    @staticmethod
    def forward(ctx, X, Z):
        X, Z = _c(X), _c(Z)
        d = cdist(X, Z)
        ctx.save_for_backward(X, Z)
        return d * d

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        X, Z = ctx.saved_tensors
        g = _c(g)
        gX = gZ = None
        if ctx.needs_input_grad[0]:      # 2 (x_i sum_j g_ij - sum_j g_ij z_j)
            gX = 2 * (X * g.sum(1, keepdim=True) - gemm(g.unsqueeze(0), Z.unsqueeze(0))[0])
        if ctx.needs_input_grad[1]:
            gZ = 2 * (Z * g.sum(0).unsqueeze(1) - gemm(g.unsqueeze(0), X.unsqueeze(0), ta=True)[0])
        return gX, gZ


def gemv(A, v, trans=False):
    """out[l] = A[l] v[l] (trans=False) or A[l]^T v[l]; A: (L, rows, cols), v: (L, cols) or (L, rows)."""
    A, v = _c(A), _c(v)
    L, rows, cols = A.shape
    out = torch.empty((L, cols if trans else rows), dtype=A.dtype, device=A.device)
    call("gemv", A.dtype, int(trans), A, v, out, rows, cols, L)
    return out


def tri_op(X, mode, out=None):
    if out is None:
        out = torch.empty_like(X)
    call("tri_op", X.dtype, X, out, X.shape[-1], X.shape[0], mode)
    return out


# ------------------------------------------------------------------------------------------------
# K1
# ------------------------------------------------------------------------------------------------
def _check_kernel_args(x1, x2, sigma, ls, a, r2, g1, g2):
    """The C ABI takes raw pointers: every floating-point argument must share x1's dtype and device, group labels must be
    int64 inside [0, n_groups) (they index the r^2 table in shared memory).  The range check is one small reduction on the
    device and is skipped with the other synchronising checks (`set_sync_checks(False)`)."""
    for name, t in (("x2", x2), ("sigma", sigma), ("lengthscale", ls), ("group coefficient", a), ("group r^2 table", r2)):
        if t is not None and (t.dtype != x1.dtype or t.device != x1.device):
            raise _cabi.GpzError(f"kernel build: {name} is {t.dtype} on {t.device}, expected {x1.dtype} on {x1.device}")
    if ls.dim() == 2:           # per-dimension (ARD) lengthscales: L x D, no groups
        if tuple(ls.shape) != (sigma.numel(), x1.shape[1]):
            raise _cabi.GpzError(f"kernel build: ARD lengthscale is {tuple(ls.shape)}, expected (L, D) = "
                                 f"{(sigma.numel(), x1.shape[1])}")
        if g1 is not None:
            raise _cabi.GpzError("kernel build: per-dimension (ARD) lengthscales have no multi-group form")
    if g1 is not None:
        g1 = g1.to(device=x1.device, dtype=torch.int64)
        g2 = g2.to(device=x1.device, dtype=torch.int64)
        if g1.numel() != x1.shape[0] or g2.numel() != x2.shape[0]:
            raise _cabi.GpzError("kernel build: one group label per point is required")
        if SYNC_CHECKS and g1.numel() and g2.numel():
            lo = min(int(g1.min()), int(g2.min()))
            hi = max(int(g1.max()), int(g2.max()))
            if lo < 0 or hi >= r2.shape[0]:
                raise IndexError(f"group label out of range [0, {r2.shape[0]}): min {lo}, max {hi}")
    return a, r2, g1, g2


def _kernel_args(x1, x2, sigma, ls, a, r2, g1, g2, check=True):
    """The leading arguments of every gpz_kernel_build_* call: ((x1, x2, sigma, ls, a, r2, g1, g2), (n1, n2, D, L, ng)), with
    a = r2 = g1 = g2 = None and ng = 0 when there are no groups (g1 None).  A 2-D ls (L x D) selects the per-dimension (ARD)
    calls gpz_kernel_build_ard_*, which take (x1, x2, sigma, ls) and the sizes without ng.  `check` makes the tensors
    contiguous and runs `_check_kernel_args`; the backward passes check=False, its tensors being the ones its forward returned
    from here."""
    if check:
        x1, x2, sigma, ls = _c(x1), _c(x2), _c(sigma), _c(ls)
        a, r2, g1, g2 = _check_kernel_args(x1, x2, sigma, ls, a, r2, g1, g2)
        if g1 is not None:
            a, r2, g1, g2 = _c(a), _c(r2), _c(g1), _c(g2)
    if g1 is None:
        a = r2 = g2 = None
    n1, D = x1.shape
    return (x1, x2, sigma, ls, a, r2, g1, g2), (n1, x2.shape[0], D, sigma.numel(), 0 if g1 is None else r2.shape[0])


class KernelBuild(Function):
    """K[l,i,j] = sigma_l^2 exp(-0.5 |x1_i-x2_j|^2/(ls_l^2 den)) / den^p_half (+ jitter on i==j); the other kinds and, for an
    L x D ls, per-dimension lengthscales as in include/gpzoo_b200.h.

    Replaces kernels.py:114-130 / 141-155 / 172-191 / 204-228 (+ utilities.py:407-418 add_jitter)."""

    @staticmethod
    def forward(ctx, x1, x2, sigma, ls, a, r2, g1, g2, p_half, jitter, want_lo=False, kind=0):
        t, (n1, n2, D, L, ng) = _kernel_args(x1, x2, sigma, ls, a, r2, g1, g2)
        dt = x1.dtype
        out = torch.empty((L, n1, n2), dtype=dt, device=x1.device)
        want_lo = bool(want_lo) and dt == torch.float32
        out_lo = torch.empty_like(out) if want_lo else None
        if ls.dim() == 2:
            call("kernel_build_ard_fwd", dt, *t[:4], n1, n2, D, L, int(kind), jitter, out, out_lo)
        else:
            call("kernel_build_fwd", dt, *t, n1, n2, D, L, ng, int(kind), p_half, jitter, out, out_lo)
        ctx.save_for_backward(*t)
        ctx.p_half = p_half
        ctx.kind = int(kind)
        ctx.want_lo = want_lo
        ctx.set_materialize_grads(False)      # no zero-filled "gradient" tensors for the non-differentiable lo plane
        if want_lo:
            ctx.mark_non_differentiable(out_lo)
            return out, out_lo
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, G, *unused):
        if G is None:
            return (None,) * 12
        grads = _kernel_build_bwd(*ctx.saved_tensors, ctx.p_half, ctx.kind, ctx.needs_input_grad[:2], G)
        return grads + (None,) * 7


def _kernel_build_bwd(x1, x2, sigma, ls, a, r2, g1, g2, p_half, kind, need, G):
    """(dL/dx1, dL/dx2, dL/dsigma, dL/dlengthscale, dL/da) from dL/dK on the current stream (csrc/kernel_build.cu)."""
    t, (n1, n2, D, L, ng) = _kernel_args(x1, x2, sigma, ls, a, r2, g1, g2, check=False)
    x1, x2, sigma, ls, a, _, g1, _ = t
    dt = x1.dtype
    G = _c(G)
    g_x1 = torch.empty_like(x1) if need[0] else None
    g_x2 = torch.empty_like(x2) if need[1] else None
    g_sigma = torch.empty_like(sigma)
    g_ls = torch.empty_like(ls)
    g_a = torch.empty_like(a) if g1 is not None else None
    if ls.dim() == 2:
        ws = torch.empty(L + L * D + n1 * D, dtype=torch.float64, device=x1.device)
        call("kernel_build_ard_bwd", dt, x1, x2, sigma, ls, n1, n2, D, L, int(kind), G, g_x1, g_x2, g_sigma, g_ls, ws)
        return g_x1, g_x2, g_sigma, g_ls, None
    ws = torch.empty(3 * L + n1 * D, dtype=torch.float64, device=x1.device)
    call("kernel_build_bwd", dt, *t, n1, n2, D, L, ng, int(kind), p_half, G, g_x1, g_x2, g_sigma, g_ls, g_a, ws)
    return g_x1, g_x2, g_sigma, g_ls, g_a


class KernelBuildBox:
    """Hand-over between KernelBuildH and the consumer of its planes (SvgpMomentsH).  The consumer's backward launches the
    kernel-build backward ITSELF on the side stream, as soon as dL/dKzx exists (so it overlaps the M x M x M chain backward that
    follows on the main stream, and dL/dKzx stays a resident workspace instead of a 4 L M N-byte tensor handed across streams
    through the autograd engine, whose deferred cross-stream frees made the allocator grow for a dozen steps); the gradients
    wait here until autograd reaches KernelBuildH.backward, which then only returns them."""
    __slots__ = ("args", "grads", "event")

    def __init__(self):
        self.args = self.grads = self.event = None


class KernelBuildH(Function):
    """KernelBuild for the split-FP16 tensor-core path: K is written once, as the fp16 planes (Kh, Kl) with Kh + Kl ~= K * sK[l]
    (4 bytes per entry; csrc/kernel_build.cu kbuild_fwd_h_kernel).  The first output is a zero-storage stand-in with K's shape
    whose only job is to carry dL/dK back to `gpz_kernel_build_bwd` (which recomputes K and never needed it stored)."""

    @staticmethod
    def forward(ctx, x1, x2, sigma, ls, a, r2, g1, g2, p_half, jitter, kind=0, box=None):
        dt = x1.dtype
        assert dt == torch.float32
        t, (n1, n2, D, L, ng) = _kernel_args(x1, x2, sigma, ls, a, r2, g1, g2)
        Kh, Kl = _plane_pair(L, n1, n2, x1.device)
        sK = torch.empty(L, dtype=dt, device=x1.device)
        if ls.dim() == 2:
            call("kernel_build_ard_fwd_h", dt, *t[:4], n1, n2, D, L, int(kind), jitter, Kh, Kl, sK)
        else:
            call("kernel_build_fwd_h", dt, *t, n1, n2, D, L, ng, int(kind), p_half, jitter, Kh, Kl, sK)
        ctx.save_for_backward(*t)
        ctx.p_half = p_half
        ctx.kind = int(kind)
        ctx.box = box
        if box is not None:
            box.args = (*t, p_half, int(kind), tuple(ctx.needs_input_grad[:2]))
        handle = torch.empty(1, dtype=dt, device=x1.device).expand(L, n1, n2)
        ctx.set_materialize_grads(False)      # otherwise autograd zero-fills "gradients" for the fp16 planes (2 x 0.67 GB)
        ctx.mark_non_differentiable(Kh, Kl, sK)
        return handle, Kh, Kl, sK

    @staticmethod
    @once_differentiable
    def backward(ctx, G, *unused):
        box = ctx.box
        if box is not None and box.grads is not None:
            grads, box.grads = box.grads, None
            torch.cuda.current_stream().wait_event(box.event)
            if G is not None and any(st != 0 for st in G.stride()):
                # dL/dK also arrived through the graph (the stand-in had a second consumer): the consumer's token is zero, so G
                # is exactly that remainder
                extra = KernelBuild.backward(ctx, G)[:5]
                grads = tuple(g if e is None else (e if g is None else g + e) for g, e in zip(grads, extra))
            return grads + (None,) * 7
        return KernelBuild.backward(ctx, G)[:12]


def cdist(x1, x2):
    """Euclidean distance matrix by direct differences (kernels.py:118 torch.cdist; no gradient)."""
    x1, x2 = _c(x1.detach()), _c(x2.detach())
    out = torch.empty((x1.shape[0], x2.shape[0]), dtype=x1.dtype, device=x1.device)
    call("cdist", x1.dtype, x1, x2, out, x1.shape[0], x2.shape[0], x1.shape[1])
    return out


# ------------------------------------------------------------------------------------------------
# K2
# ------------------------------------------------------------------------------------------------
class CholeskyInverse(Function):
    """(Lc, Linv) = (chol(Kzz), chol(Kzz)^-1) for Kzz (L x M x M).  gp.py:213 torch.linalg.cholesky; the
    inverse factor turns cholesky_solve (gp.py:218) and kl_divergence's solves into triangular products."""

    @staticmethod
    def forward(ctx, Kzz):
        dt = Kzz.dtype
        L, M, _ = Kzz.shape
        W = Kzz.detach().clone(memory_format=torch.contiguous_format)
        info = torch.empty(L, dtype=torch.int32, device=Kzz.device)
        Lc, Linv, tmp = torch.empty_like(W), torch.empty_like(W), torch.empty_like(W)
        if USE_TENSOR_CORES and dt == torch.float32 and M > CHOL_TC_MIN_M and M % 4 == 0:
            lo_ws = torch.empty((4,) + tuple(W.shape), dtype=dt, device=W.device)      # lo planes shadowing W, Lc, Linv, tmp
            call("chol_inv_tc", dt, W, Lc, Linv, tmp, lo_ws, M, L, info)
        else:
            call("chol_inv", dt, W, Lc, Linv, tmp, M, L, info)
        _track_info(info)
        if SYNC_CHECKS:
            check_cholesky_info()
        ctx.save_for_backward(Lc, Linv)
        return Lc, Linv

    @staticmethod
    @once_differentiable
    def backward(ctx, gLc, gLinv):
        Lc, Linv = ctx.saved_tensors
        if gLc is None and gLinv is None:
            return None
        g = tri_op(_c(gLc), 2) if gLc is not None else torch.zeros_like(Lc)
        if gLinv is not None:
            t1 = gemm(Linv, _c(gLinv), ta=True, a_tri=2)                       # Linv^T gLinv
            gemm(t1, Linv, tb=True, alpha=-1.0, beta=1.0, out=g, b_tri=2, d_tri=1)   # g -= tril(t1 Linv^T)
        P = gemm(Lc, g, ta=True, a_tri=2, b_tri=1, d_tri=1)                    # tril(Lc^T g)
        tri_op(P, 0, out=P)                                                    # halve the diagonal
        t1 = gemm(Linv, P, ta=True, a_tri=2, b_tri=1)                          # Linv^T Phi
        t2 = gemm(t1, Linv, b_tri=1)                                           # ... Linv
        return tri_op(t2, 1)                                                   # symmetrise


def chain_ok(dtype, M):
    """fp32 chains large enough for the fused two-call implementation (csrc/chain.cu)."""
    return (USE_TENSOR_CORES and FUSED_CHAIN and dtype == torch.float32
            and bool(_cabi.lib().gpz_svgp_chain_supported(int(M))))


class SvgpChain(Function):
    """Everything between the jittered Kzz and the whitened operands of the predictive kernels, as ONE forward and ONE backward
    C-ABI call (csrc/chain.cu): (Lc, Linv) = chol_inv(Kzz), Lu = lower_cholesky(raw), T = Linv Lu, q = Linv mu and
    kl = KL(N(mu, Lu Lu^T) || N(0, Lc Lc^T)) per factor.  Replaces CholeskyInverse + LowerCholesky + Whiten + MvnKL (and the
    ATen gradient accumulation between them) for fp32 models with M >= 128.  `consume`: Kzz may be overwritten."""

    @staticmethod
    def forward(ctx, Kzz, Lu_raw, mu, consume):
        L, M, _ = Kzz.shape
        dt = Kzz.dtype
        dev = Kzz.device
        W = _c(Kzz.detach())
        if W.data_ptr() == Kzz.data_ptr() and not consume:
            W = W.clone()
        Lu_raw, mu = _c(Lu_raw.detach()), _c(mu.detach())
        chol_tc = int(M > CHOL_TC_MIN_M)
        Lc, Linv, Lu, T = (torch.empty((L, M, M), dtype=dt, device=dev) for _ in range(4))
        q = torch.empty((L, M), dtype=dt, device=dev)
        kl = torch.empty(L, dtype=dt, device=dev)
        aux = torch.empty((6, L, M, M), dtype=dt, device=dev)
        ws = torch.empty(((5 if chol_tc else 1) * L * M * M + 4 * L,), dtype=dt, device=dev)
        info = torch.empty(L, dtype=torch.int32, device=dev)
        call("svgp_chain_fwd", dt, W, Lu_raw, mu, Lc, Linv, Lu, T, q, kl, aux, ws, M, L, chol_tc, info)
        _track_info(info)
        if SYNC_CHECKS:
            check_cholesky_info()
        ctx.save_for_backward(Lc, Linv, Lu, T, q, mu, aux)
        ctx.set_materialize_grads(False)
        return Lc, Linv, Lu, T, q, kl

    @staticmethod
    @once_differentiable
    def backward(ctx, gLc, gLinv, gLu, gT, gq, gkl):
        Lc, Linv, Lu, T, q, mu, aux = ctx.saved_tensors
        L, M, _ = Lc.shape
        dt, dev = Lc.dtype, Lc.device
        cc = lambda t: None if t is None else _c(t)
        gLc, gLinv, gLu, gT, gq, gkl = cc(gLc), cc(gLinv), cc(gLu), cc(gT), cc(gq), cc(gkl)
        gKzz = torch.empty((L, M, M), dtype=dt, device=dev)
        gLu_raw = torch.empty_like(gKzz)
        gmu = torch.empty((L, M), dtype=dt, device=dev)
        grp = _chain_shard_group
        if grp is not None and torch.distributed.get_world_size(grp) > 1 and gLc is None and gLu is None:
            return SvgpChain._backward_sharded(grp, ctx.saved_tensors, gLinv, gT, gq, gkl, gKzz, gLu_raw, gmu) + (None,)
        ws = torch.empty((12 * L * M * M + 2 * L * M,), dtype=dt, device=dev)
        call("svgp_chain_bwd", dt, Lc, Linv, Lu, T, q, mu, aux, gLc, gLinv, gLu, gT, gq, gkl, gKzz, gLu_raw, gmu, ws, M, L)
        return gKzz, gLu_raw, gmu, None

    @staticmethod
    def _backward_sharded(grp, saved, gLinv, gT, gq, gkl, gKzz, gLu_raw, gmu):
        """Data-parallel ranks hold PARTIAL gradients (sums over their own spots) of the replicated chain's outputs.  The chain's
        backward is linear in them, so instead of every rank pushing its partials through all L factors (and the all-reduce
        summing the results) the partials are summed FIRST, factor by factor onto the rank that owns the factor (one all-to-all
        + a sum over the senders), and each rank runs the backward of its own factors only.  It returns zeros for the factors
        it does not own; the step's gradient all-reduce then assembles the totals exactly as before.  The replicated O(M^3)
        backward (7 GEMMs per factor) shrinks from L to ceil(L / world) factors per rank."""
        import torch.distributed as dist
        Lc, Linv, Lu, T, q, mu, aux = saved
        L, M, _ = Lc.shape
        dt, dev = Lc.dtype, Lc.device
        world, rank = dist.get_world_size(grp), dist.get_rank(grp)
        bounds = [(r * L) // world for r in range(world + 1)]              # contiguous blocks of factors, sizes differ by <= 1
        l0, l1 = bounds[rank], bounds[rank + 1]
        own = l1 - l0
        zeros = lambda *shape: torch.zeros(shape, dtype=dt, device=dev)
        gLinv = gLinv if gLinv is not None else zeros(L, M, M)
        gT = gT if gT is not None else zeros(L, M, M)
        gq = gq if gq is not None else zeros(L, M)
        # one flat buffer per factor: [gLinv_l | gT_l | gq_l]
        per = 2 * M * M + M
        send = torch.empty((L, per), dtype=dt, device=dev)
        send[:, :M * M] = gLinv.reshape(L, -1)
        send[:, M * M:2 * M * M] = gT.reshape(L, -1)
        send[:, 2 * M * M:] = gq
        recv = torch.empty((world, own, per), dtype=dt, device=dev)
        dist.all_to_all_single(recv.view(-1), send.view(-1), output_split_sizes=[own * per] * world,
                               input_split_sizes=[(bounds[r + 1] - bounds[r]) * per for r in range(world)], group=grp)
        gKzz.zero_(), gLu_raw.zero_(), gmu.zero_()
        if own > 0:
            tot = recv.sum(0)                                              # partials of every rank, own factors
            gLinv_o = tot[:, :M * M].reshape(own, M, M).contiguous()
            gT_o = tot[:, M * M:2 * M * M].reshape(own, M, M).contiguous()
            gq_o = tot[:, 2 * M * M:].contiguous()
            # every rank weighted the KL by 1 / world (kl_weight): the owner applies the full weight
            gkl_o = (gkl[l0:l1] * world).contiguous() if gkl is not None else None
            sl = lambda t: t[l0:l1].contiguous()
            aux_o = aux[:, l0:l1].contiguous()
            gK_o = torch.empty((own, M, M), dtype=dt, device=dev)
            gLu_o = torch.empty_like(gK_o)
            gmu_o = torch.empty((own, M), dtype=dt, device=dev)
            ws = torch.empty((12 * own * M * M + 2 * own * M,), dtype=dt, device=dev)
            call("svgp_chain_bwd", dt, sl(Lc), sl(Linv), sl(Lu), sl(T), sl(q), sl(mu), aux_o, None, gLinv_o, None, gT_o, gq_o,
                 gkl_o, gK_o, gLu_o, gmu_o, ws, M, own)
            gKzz[l0:l1], gLu_raw[l0:l1], gmu[l0:l1] = gK_o, gLu_o, gmu_o
        return gKzz, gLu_raw, gmu


_chain_shard_group = None


def set_chain_sharding(group):
    """Data-parallel training: shard the backward of the replicated O(M^3) chain by factor over `group` (a torch.distributed
    process group; None turns it off).  Requires that every rank of the group calls the step with the same parameters and a
    KL weight of 1 / world_size, and that the shared-parameter gradients are summed over the group afterwards
    (`gpzoo_b200.distributed.FlatGradReducer`)."""
    global _chain_shard_group
    _chain_shard_group = group


def fused_moments_ok(dtype, M, N):
    """fp32 problems that take the fused chain + split-FP16 predict Function with the merged backward."""
    return FUSED_MOMENTS and chain_ok(dtype, M) and predict_h_ok(dtype, M, N)


class SvgpMomentsH(Function):
    """SvgpChain + PredictH as ONE autograd node (fp32): jittered Kzz, raw Lu, mu and the fp16 planes of Kzx ->
    predictive mean / variance, per-factor KL, Lc and Lu.  Keeping Linv, T and q internal is what allows the MERGED backward
    (csrc/chain.cu gpz_svgp_chain_bwd_s1): one reduction over the spots (S1 = A diag(2 gv) A^T) and 8 M x M x M products instead
    of two reductions and 11 products."""

    @staticmethod
    def forward(ctx, Kzz, Lu_raw, mu, Kxx, Kzx, Kh, Kl, sK, consume, box=None):
        L, M, _ = Kzz.shape
        dt, dev = Kzz.dtype, Kzz.device
        N = Kh.shape[-1]
        W = _c(Kzz.detach())
        if W.data_ptr() == Kzz.data_ptr() and not consume:
            W = W.clone()
        Lu_raw, mu, Kxx, Kh, Kl, sK = _c(Lu_raw.detach()), _c(mu.detach()), _c(Kxx.detach()), _c(Kh), _c(Kl), _c(sK)
        chol_tc = int(M > CHOL_TC_MIN_M)
        Lc, Linv, Lu, T = (torch.empty((L, M, M), dtype=dt, device=dev) for _ in range(4))
        q = torch.empty((L, M), dtype=dt, device=dev)
        kl = torch.empty(L, dtype=dt, device=dev)
        aux = torch.empty((6, L, M, M), dtype=dt, device=dev)
        ws = torch.empty(((5 if chol_tc else 1) * L * M * M + 4 * L,), dtype=dt, device=dev)
        info = torch.empty(L, dtype=torch.int32, device=dev)
        call("svgp_chain_fwd", dt, W, Lu_raw, mu, Lc, Linv, Lu, T, q, kl, aux, ws, M, L, chol_tc, info)
        _track_info(info)
        (Ah, Al), (Ch, Cl) = _plane_pair(L, M, N, dev), _plane_pair(L, M, N, dev)
        mean = torch.empty((L, N), dtype=dt, device=dev)
        var = torch.empty_like(mean)
        ws_h = torch.empty(8 * L * M * M, dtype=torch.float16, device=dev)
        ws_f = torch.empty(2 * L * N + 16 * L, dtype=dt, device=dev)
        call("svgp_predict_fwd_h", dt, Kh, Kl, sK, Linv, T, q, Kxx, Ah, Al, Ch, Cl, mean, var, ws_h, ws_f, M, N, L)
        st = ws_f[2 * L * N:].view(-1, L)
        r_sA, r_aA, r_aC, r_sC = (_stat_row(i) for i in (0, 1, 2, 5))
        _track_amax(torch.stack((st[r_aA], st[r_aC])), torch.stack((st[r_sA], st[r_sC])), ("A", "C"))
        if SYNC_CHECKS:
            check_cholesky_info()
        ctx.save_for_backward(Lc, Linv, Lu, T, q, mu, aux, Kh, Kl, sK, Ah, Al, Ch, Cl, ws_h, ws_f)
        ctx.set_materialize_grads(False)
        ctx.box = box
        return mean, var, kl, Lc, Lu

    @staticmethod
    @once_differentiable
    def backward(ctx, gm, gv, gkl, gLc, gLu):
        Lc, Linv, Lu, T, q, mu, aux, Kh, Kl, sK, Ah, Al, Ch, Cl, ws_h, ws_f = ctx.saved_tensors
        L, M, N = Kh.shape
        dt, dev = Lc.dtype, Lc.device
        cc = lambda t: None if t is None else _c(t)
        gm = _c(gm) if gm is not None else torch.zeros((L, N), dtype=dt, device=dev)
        gv = _c(gv) if gv is not None else torch.zeros((L, N), dtype=dt, device=dev)
        gkl, gLc, gLu = cc(gkl), cc(gLc), cc(gLu)
        AWh, AWl, gAh, gAl = _workspace("predict_bwd_planes", (4, L, M, N), torch.float16, dev)
        box = ctx.box
        early = box is not None and box.args is not None and ctx.needs_input_grad[4]
        main = torch.cuda.current_stream()
        if early:
            # dL/dKzx never leaves this call: resident workspace, read by the kernel-build backward launched below on the side stream
            gKzx = _workspace("moments_gKzx", (L, M, N), dt, dev)
            wkey = ("moments_gKzx", main.cuda_stream)
            if wkey in _workspace_readers:
                main.wait_event(_workspace_readers[wkey])             # the previous step's reader (side stream) is done with it
        else:
            gKzx = torch.empty((L, M, N), dtype=dt, device=dev) if ctx.needs_input_grad[4] else _workspace(
                "moments_gKzx", (L, M, N), dt, dev)
        gqp = torch.empty((L, M), dtype=dt, device=dev)
        S = _workspace("moments_bwd_S", (2, L, M, M), dt, dev)              # S1 and its lo plane
        call("svgp_predict_bwd_h", dt, Kh, Kl, sK, T, q, Ah, Al, Ch, Cl, gm, gv, AWh, AWl, gAh, gAl, gKzx, None, None, gqp, ws_h,
             ws_f, S, M, N, L)
        stt = ws_f[2 * L * N:].view(-1, L)
        _track_amax(stt[_stat_row(4)].unsqueeze(0), stt[_stat_row(3)].unsqueeze(0), ("dL/dA",))
        if early:
            side = side_stream(dev)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                box.grads = _kernel_build_bwd(*box.args, gKzx)
                box.event = torch.cuda.Event()
                box.event.record(side)
            _workspace_readers[wkey] = box.event
            g_handle = torch.zeros(1, dtype=dt, device=dev).expand(L, M, N)   # zero token: KernelBuildH.backward returns box.grads
        else:
            g_handle = gKzx if ctx.needs_input_grad[4] else None
        gKzz = torch.empty((L, M, M), dtype=dt, device=dev)
        gLu_raw = torch.empty_like(gKzz)
        gmu = torch.empty((L, M), dtype=dt, device=dev)
        ws = _workspace("chain_bwd_s1_ws", (13 * L * M * M + 2 * L * M,), dt, dev)
        call("svgp_chain_bwd_s1", dt, Lc, Linv, Lu, T, q, mu, aux, S[0], S[1], gqp, gkl, gLc, gLu, gKzz, gLu_raw, gmu, ws, M, L)
        return gKzz, gLu_raw, gmu, gv, g_handle, None, None, None, None, None


class LowerCholesky(Function):
    """transform_to(constraints.lower_cholesky) (gp.py:220): tril(raw,-1) + diag(exp(diag raw))."""

    @staticmethod
    def forward(ctx, raw):
        raw = _c(raw)
        out = torch.empty_like(raw)
        call("lower_cholesky_fwd", raw.dtype, raw, out, raw.shape[-1], raw.shape[0])
        ctx.save_for_backward(out)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        (out,) = ctx.saved_tensors
        g = _c(g)
        graw = torch.empty_like(g)
        call("lower_cholesky_bwd", g.dtype, g, out, graw, g.shape[-1], g.shape[0])
        return graw


class Whiten(Function):
    """T = Linv Lu (lower), q = Linv mu — the quantities torch computes with solve_triangular inside
    kl_divergence(qU, pU) (torch kl.py) and that the predictive variance needs as Lu^T Lc^-T."""

    @staticmethod
    def forward(ctx, Linv, Lu, mu):
        Linv, Lu, mu = _c(Linv), _c(Lu), _c(mu)
        T = gemm(Linv, Lu, a_tri=1, b_tri=1, d_tri=1)
        q = gemv(Linv, mu)
        ctx.save_for_backward(Linv, Lu, mu)
        return T, q

    @staticmethod
    @once_differentiable
    def backward(ctx, gT, gq):
        Linv, Lu, mu = ctx.saved_tensors
        gLinv = torch.zeros_like(Linv)
        gLu = gmu = None
        if gT is not None:
            gT = _c(gT)
            gemm(gT, Lu, tb=True, out=gLinv, b_tri=2, d_tri=1)
            gLu = gemm(Linv, gT, ta=True, a_tri=2, d_tri=1)
        if gq is not None:
            gq = _c(gq).unsqueeze(-1)
            gemm(gq, mu.unsqueeze(-1), tb=True, beta=1.0, out=gLinv, d_tri=1)
            gmu = gemv(Linv, gq.squeeze(-1), trans=True)
        return gLinv, gLu, gmu


# ------------------------------------------------------------------------------------------------
# K3 / K4
# ------------------------------------------------------------------------------------------------
def tensor_core_predict_ok(dtype, M, N):
    return (USE_TENSOR_CORES and dtype == torch.float32
            and bool(_cabi.lib().gpz_svgp_predict_tc_supported(int(M), int(N))))


class Predict(Function):
    """SVGP predictive mean and variance (gp.py:218-225 + utilities.py:382-397), see csrc/predict.cu.
    fp32 with Kzx_lo given: tcgen05 split-TF32 GEMMs (csrc/umma_gemm.cu); otherwise exact CUDA-core GEMMs."""

    @staticmethod
    def forward(ctx, Kxx, Kzx, Linv, T, q, Kzx_lo=None):
        Kxx, Kzx, Linv, T, q = _c(Kxx), _c(Kzx), _c(Linv), _c(T), _c(q)
        dt = Kzx.dtype
        L, M, N = Kzx.shape
        A = torch.empty_like(Kzx)
        C = torch.empty_like(Kzx)
        mean = torch.empty((L, N), dtype=dt, device=Kzx.device)
        var = torch.empty_like(mean)
        tc = Kzx_lo is not None and tensor_core_predict_ok(dt, M, N)
        ctx.tc = tc
        if tc:
            Kzx_lo = _c(Kzx_lo)
            A_lo = torch.empty_like(Kzx)
            ws = torch.empty(6 * L * M * M + 2 * L * N, dtype=dt, device=Kzx.device)
            call("svgp_predict_fwd_tc", dt, Kzx, Kzx_lo, Linv, T, q, Kxx, A, A_lo, C, mean, var, ws, M, N, L)
            ctx.save_for_backward(Kzx, Linv, T, q, A, C, Kzx_lo, A_lo, ws)
        else:
            call("svgp_predict_fwd", dt, Kzx, Linv, T, q, Kxx, A, C, mean, var, M, N, L)
            ctx.save_for_backward(Kzx, Linv, T, q, A, C)
        return mean, var

    @staticmethod
    @once_differentiable
    def backward(ctx, gm, gv):
        if ctx.tc:
            Kzx, Linv, T, q, A, C, Kzx_lo, A_lo, ws = ctx.saved_tensors
        else:
            Kzx, Linv, T, q, A, C = ctx.saved_tensors
        dt = Kzx.dtype
        L, M, N = Kzx.shape
        gm = _c(gm) if gm is not None else torch.zeros((L, N), dtype=dt, device=Kzx.device)
        gv = _c(gv) if gv is not None else torch.zeros((L, N), dtype=dt, device=Kzx.device)
        # the kernels turn their C argument into gC in place: hand them a copy, the saved tensor must survive for a second
        # backward over the same graph (retain_graph=True)
        C = C.clone()
        gA = torch.empty_like(Kzx)
        gKzx = torch.empty_like(Kzx)
        gLinv = torch.zeros_like(Linv)
        gT = torch.zeros_like(T)
        gq = torch.empty_like(q)
        if ctx.tc:
            C_lo = torch.empty_like(Kzx)
            gA_lo = torch.empty_like(Kzx)
            call("svgp_predict_bwd_tc", dt, Kzx, Kzx_lo, Linv, T, q, A, A_lo, C, C_lo, gm, gv, gA, gA_lo, gKzx, gLinv, gT, gq, ws,
                 M, N, L)
        else:
            call("svgp_predict_bwd", dt, Kzx, Linv, T, q, A, C, gm, gv, gA, gKzx, gLinv, gT, gq, M, N, L)
        return gv, gKzx, gLinv, gT, gq, None


def predict_h_ok(dtype, M, N):
    """fp32 problems large and aligned enough for the split-FP16 tcgen05 path."""
    return (USE_TENSOR_CORES and TENSOR_CORE_ARITH == "fp16x3" and dtype == torch.float32
            and bool(_cabi.lib().gpz_svgp_predict_h_supported(int(M), int(N))))


def _stat_row(which):
    return int(_cabi.lib().gpz_svgp_predict_h_stat_row(which))


class PredictH(Function):
    """Predict on fp16 operand planes (split-FP16 tcgen05 GEMMs, csrc/predict.cu predict_fwd_h / predict_bwd_h).
    `Kzx` is KernelBuildH's stand-in (it only routes dL/dKzx); (Kh, Kl, sK) are the planes it wrote."""

    @staticmethod
    def forward(ctx, Kxx, Kzx, Linv, T, q, Kh, Kl, sK):
        Kxx, Linv, T, q, Kh, Kl, sK = _c(Kxx), _c(Linv), _c(T), _c(q), _c(Kh), _c(Kl), _c(sK)
        dt = Linv.dtype
        L, M, N = Kh.shape
        dev = Kh.device
        (Ah, Al), (Ch, Cl) = _plane_pair(L, M, N, dev), _plane_pair(L, M, N, dev)
        mean = torch.empty((L, N), dtype=dt, device=dev)
        var = torch.empty_like(mean)
        ws_h = torch.empty(8 * L * M * M, dtype=torch.float16, device=dev)
        ws_f = torch.empty(2 * L * N + 16 * L, dtype=dt, device=dev)
        call("svgp_predict_fwd_h", dt, Kh, Kl, sK, Linv, T, q, Kxx, Ah, Al, Ch, Cl, mean, var, ws_h, ws_f, M, N, L)
        ctx.save_for_backward(Kh, Kl, sK, Linv, T, q, Ah, Al, Ch, Cl, ws_h, ws_f)
        # tracked max |A|, max |C| (slots 7, 8 of the stats block, csrc/predict.cu): examined lazily with the Cholesky info
        st = ws_f[2 * L * N:].view(-1, L)
        r_sA, r_aA, r_aC, r_sC = (_stat_row(i) for i in (0, 1, 2, 5))
        _track_amax(torch.stack((st[r_aA], st[r_aC])), torch.stack((st[r_sA], st[r_sC])), ("A", "C"))
        if SYNC_CHECKS:
            check_cholesky_info()
        return mean, var

    @staticmethod
    @once_differentiable
    def backward(ctx, gm, gv):
        Kh, Kl, sK, Linv, T, q, Ah, Al, Ch, Cl, ws_h, ws_f = ctx.saved_tensors
        dt = Linv.dtype
        L, M, N = Kh.shape
        dev = Kh.device
        gm = _c(gm) if gm is not None else torch.zeros((L, N), dtype=dt, device=dev)
        gv = _c(gv) if gv is not None else torch.zeros((L, N), dtype=dt, device=dev)
        AWh, AWl, gAh, gAl = _workspace("predict_bwd_planes", (4, L, M, N), torch.float16, dev)
        gKzx = torch.empty((L, M, N), dtype=dt, device=dev)
        gLinv = torch.zeros_like(Linv)
        gT = torch.zeros_like(T)
        gq = torch.empty_like(q)
        call("svgp_predict_bwd_h", dt, Kh, Kl, sK, T, q, Ah, Al, Ch, Cl, gm, gv, AWh, AWl, gAh, gAl, gKzx, gLinv, gT, gq, ws_h,
             ws_f, None, M, N, L)
        st = ws_f[2 * L * N:].view(-1, L)
        _track_amax(st[_stat_row(4)].unsqueeze(0), st[_stat_row(3)].unsqueeze(0), ("dL/dA",))   # max |gA| vs its scale
        return gv, gKzx, gLinv, gT, gq, None, None, None


def umma_gemm(A, B, b_kmajor, Alo=None, Blo=None, Cin=None, alpha=1.0, want_lo=False, a_tri=0, b_tri=0, d_tri=0, splitk=1,
              n_terms=3):
    """Direct access to the tcgen05 split-TF32 batched GEMM (fp32).  A: (b, m, k); B: (b, k, n) or, b_kmajor, (b, n, k)."""
    bsz, m, k = A.shape
    n = B.shape[1] if b_kmajor else B.shape[2]
    lo = lambda x: tf32_lo(x)
    if n_terms == 3:
        Alo = lo(A) if Alo is None else Alo
        Blo = lo(B) if Blo is None else Blo
    D = torch.zeros((bsz, m, n), dtype=torch.float32, device=A.device)
    Dlo = torch.empty_like(D) if want_lo else None
    call("umma_gemm", torch.float32, int(b_kmajor), m, n, k, alpha, A, Alo, A.shape[2], A.shape[1] * A.shape[2], B, Blo,
         B.shape[2], B.shape[1] * B.shape[2], Cin, D, Dlo, n, m * n, bsz, a_tri, b_tri, d_tri, splitk, n_terms)
    return (D, Dlo) if want_lo else D


def split16(x, transpose=False):
    """fp16 operand planes of a batch of fp32 matrices for the split-FP16 GEMM: (hi, lo, scale) with hi + lo ~= x * scale[b]
    (22 significant bits) and scale[b] the power of two that puts max |x[b]| in (2^14, 2^15].  transpose=True also returns the
    planes of the per-matrix transposes: (hi, lo, hiT, loT, scale)."""
    x = _c(x)
    bsz, rows, cols = x.shape
    h = torch.empty((bsz, rows, cols), dtype=torch.float16, device=x.device)
    l = torch.empty_like(h)
    hT = torch.empty((bsz, cols, rows), dtype=torch.float16, device=x.device) if transpose else None
    lT = torch.empty_like(hT) if transpose else None
    scale = torch.empty(bsz, dtype=torch.float32, device=x.device)
    ws = torch.empty(bsz, dtype=torch.int32, device=x.device)
    call("split16", torch.float32, x, rows, cols, bsz, h, l, hT, lT, scale, ws)
    return (h, l, hT, lT, scale) if transpose else (h, l, scale)


def umma_gemm16(A, B, b_kmajor, a_tri=0, b_tri=0, d_tri=0, splitk=1, n_terms=3, alpha=1.0, out_planes=False, out_scale=None,
                want_amax=False, Cin=None, out=None):
    """Direct access to the tcgen05 split-FP16 batched GEMM.  A = (hi, lo, scale) planes of (b, m, k); B = planes of (b, k, n) or,
    b_kmajor, (b, n, k).  Returns fp32 D, or with out_planes the fp16 planes (Dh, Dl) of D * out_scale; want_amax adds max |D|."""
    Ah, Al, sa = A
    Bh, Bl, sb = B
    bsz, m, k = Ah.shape
    n = Bh.shape[1] if b_kmajor else Bh.shape[2]
    dev = Ah.device
    D = None if out_planes else (out if out is not None else torch.zeros((bsz, m, n), dtype=torch.float32, device=dev))
    Dh = torch.zeros((bsz, m, n), dtype=torch.float16, device=dev) if out_planes else None
    Dl = torch.zeros_like(Dh) if out_planes else None
    amax = torch.zeros(bsz, dtype=torch.int32, device=dev) if want_amax else None
    call("umma_gemm16", torch.float32, int(b_kmajor), m, n, k, alpha, Ah, Al, Ah.shape[2], Ah.shape[1] * Ah.shape[2], sa, Bh, Bl,
         Bh.shape[2], Bh.shape[1] * Bh.shape[2], sb, Cin, D, Dh, Dl, out_scale, amax, n, m * n, bsz, a_tri, b_tri, d_tri, splitk,
         n_terms)
    res = (Dh, Dl) if out_planes else D
    return (res, amax.view(torch.float32)) if want_amax else res


# (x, lo) planes and transposes of the M x M operands are needed by several GEMMs of one step (Linv: whitening, predict,
# Cholesky backward ...).  They are cached per source tensor for the duration of a step; the cache holds a reference to the
# source so its memory cannot be recycled under the same key, and `clear_step_cache()` runs at the start of every step.
_step_cache = {}


def clear_step_cache():
    _step_cache.clear()


def _cached(kind, x, make):
    key = (kind, x.data_ptr(), x._version, tuple(x.shape))
    hit = _step_cache.get(key)
    if hit is None:
        if len(_step_cache) > 64:
            _step_cache.clear()
        hit = (make(), x)
        _step_cache[key] = hit
    return hit[0]


def tf32_lo(x):
    x = _c(x)

    def make():
        lo = torch.empty_like(x)
        call("tf32_lo", torch.float32, x, lo, x.numel())
        return lo
    return _cached("lo", x, make) if x.dim() == 3 and x.shape[-1] == x.shape[-2] else make()


# ------------------------------------------------------------------------------------------------
# K6  VNNGP
# ------------------------------------------------------------------------------------------------
def vnngp_neighbors(X, Z, K):
    """K nearest inducing points of every x (ascending distance, ties to the lower index) — gp.py:64."""
    X, Z = _c(X.detach()), _c(Z.detach())
    idx = torch.empty((X.shape[0], K), dtype=torch.int64, device=X.device)
    call("vnngp_neighbors", X.dtype, X, Z, idx, X.shape[0], Z.shape[0], X.shape[1], K)
    return idx


class OuterLower(Function):
    """S = Lu Lu^T (gp.py:100-102 / 221) with gLu = tril((gS + gS^T) Lu)."""

    @staticmethod
    def forward(ctx, Lu):
        Lu = _c(Lu)
        ctx.save_for_backward(Lu)
        return gemm(Lu, Lu, tb=True, a_tri=1, b_tri=2)

    @staticmethod
    @once_differentiable
    def backward(ctx, gS):
        (Lu,) = ctx.saved_tensors
        gS = _c(gS)
        g = gemm(gS, Lu, b_tri=1)
        gemm(gS, Lu, ta=True, b_tri=1, beta=1.0, out=g)
        return tri_op(g, 2)


class VnngpPredict(Function):
    """Nearest-neighbour predictive mean / variance (gp.py:67-106), one warp per point (csrc/vnngp.cu)."""

    @staticmethod
    def forward(ctx, X, Z, sigma, ls, Kzz, S, mu, Kxx, nn, jitter):
        X, Z, sigma, ls, Kzz, S, mu, Kxx = (_c(t) for t in (X, Z, sigma, ls, Kzz, S, mu, Kxx))
        dt = Kzz.dtype
        L, M, _ = Kzz.shape
        N, D = X.shape
        K = nn.shape[1]
        mean = torch.empty((L, N), dtype=dt, device=X.device)
        var = torch.empty_like(mean)
        call("vnngp_fwd", dt, X, Z, sigma, ls, Kzz, S, mu, Kxx, nn, N, M, D, L, K, jitter, mean, var)
        ctx.save_for_backward(X, Z, sigma, ls, Kzz, S, mu, Kxx, nn)
        ctx.jitter = jitter
        return mean, var

    @staticmethod
    @once_differentiable
    def backward(ctx, gm, gv):
        X, Z, sigma, ls, Kzz, S, mu, Kxx, nn = ctx.saved_tensors
        dt = Kzz.dtype
        L, M, _ = Kzz.shape
        N, D = X.shape
        K = nn.shape[1]
        gm = _c(gm) if gm is not None else torch.zeros((L, N), dtype=dt, device=X.device)
        gv = _c(gv) if gv is not None else torch.zeros((L, N), dtype=dt, device=X.device)
        gKzz, gS = torch.empty_like(Kzz), torch.empty_like(S)
        gmu, gZ = torch.empty_like(mu), torch.empty_like(Z)
        gsl = torch.empty(2 * L, dtype=torch.float64, device=X.device)
        call("vnngp_bwd", dt, X, Z, sigma, ls, Kzz, S, mu, Kxx, nn, N, M, D, L, K, ctx.jitter, gm, gv, gKzz, gS, gmu, gZ, gsl)
        return None, gZ, gsl[:L].to(dt), gsl[L:].to(dt), gKzz, gS, gmu, gv, None, None


# ------------------------------------------------------------------------------------------------
# K5
# ------------------------------------------------------------------------------------------------
class MvnKL(Function):
    """kl_divergence(MVN(mu, Lu), MVN(0, Lc)) per factor (utilities.py:481,616; torch kl.py)."""

    @staticmethod
    def forward(ctx, T, q, Lc, Lu):
        T, q, Lc, Lu = _c(T), _c(q), _c(Lc), _c(Lu)
        L, M, _ = T.shape
        kl = torch.empty(L, dtype=T.dtype, device=T.device)
        ws = torch.empty(L, dtype=torch.float64, device=T.device)
        call("mvn_kl_fwd", T.dtype, T, q, Lc, Lu, kl, ws, M, L)
        ctx.save_for_backward(T, q, Lc, Lu)
        return kl

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        T, q, Lc, Lu = ctx.saved_tensors
        L, M, _ = T.shape
        g = _c(g)
        gT, gLc, gLu, gq = torch.empty_like(T), torch.empty_like(T), torch.empty_like(T), torch.empty_like(q)
        call("mvn_kl_bwd", T.dtype, g, T, q, Lc, Lu, gT, gq, gLc, gLu, M, L)
        return gT, gq, gLc, gLu


# ------------------------------------------------------------------------------------------------
# K7
# ------------------------------------------------------------------------------------------------
class PoissonLL(Function):
    """mean_E sum_{g,n} Poisson log-lik of y under rate = softplus(V) (w(W) @ exp(mean + eps*sd)),
    with all gradients produced by the same pass (csrc/poisson.cu).  y is a dense G x N tensor or a `SparseCounts`
    (read by the K7-CSC kernel, whose work scales with the nonzeros)."""

    Y_KINDS = {torch.uint8: 1, torch.int16: 2, torch.int32: 3}     # counts stored as integers (gpz_poisson_fwdbwd_yt_f32)

    @staticmethod
    def forward(ctx, y, idx, W, V, mean, spread, eps, n_var, clamp_min, w_softplus, with_lgamma):
        W, V, mean, spread, eps = _c(W), _c(V), _c(mean), _c(spread), _c(eps)
        dt = W.dtype
        if isinstance(y, SparseCounts):
            gW, gV, gmean, gspread, ll, idx = _poisson_csc(y, idx, W, V, mean, spread, eps, n_var, clamp_min, w_softplus, with_lgamma)
            ctx.save_for_backward(gW, gV, gmean, gspread, idx)
            ctx.nV = V.shape[0]
            return ll.to(dt).reshape(())
        gW, gV, gmean, gspread, ll, idx, _ = _k7_dense(y, idx, W, V, None, mean, spread, eps, n_var, clamp_min, w_softplus, with_lgamma)
        ctx.save_for_backward(gW, gV, gmean, gspread, idx)
        ctx.nV = V.shape[0]
        return ll.to(dt).reshape(())

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        gW, gV, gmean, gspread, idx = ctx.saved_tensors
        return None, None, g * gW, g * _scatter_gV(ctx.nV, gV, idx), g * gmean, g * gspread, None, None, None, None, None


class NegBinLL(Function):
    """mean_E sum_{g,n} negative-binomial log-lik of dense counts y under the same rate as PoissonLL and the per-gene dispersion
    theta = softplus(D) (D: G, raw), with every gradient, dD included, from one pass (K7-NB, csrc/poisson.cu):
    log NB = lgamma(y + theta) - lgamma(theta) - lgamma(y + 1) + y log(r / (theta + r)) - theta log1p(r / theta)."""

    @staticmethod
    def forward(ctx, y, idx, W, V, D, mean, spread, eps, n_var, clamp_min, w_softplus, with_lgamma):
        if isinstance(y, SparseCounts):
            raise NotImplementedError(
                "the negative-binomial likelihood needs dense counts: its zero counts each contribute -theta log1p(r / theta), "
                "which has no closed form through the loadings' column sums the way the Poisson zeros' -r does, so the work is "
                "G x N whatever the density; pass y.to_dense()")
        W, V, D, mean, spread, eps = _c(W), _c(V), _c(D), _c(mean), _c(spread), _c(eps)
        assert D.shape == (W.shape[0],) and D.dtype == W.dtype
        gW, gV, gmean, gspread, ll, idx, gD = _k7_dense(y, idx, W, V, D, mean, spread, eps, n_var, clamp_min, w_softplus, with_lgamma)
        ctx.save_for_backward(gW, gV, gD, gmean, gspread, idx)
        ctx.nV = V.shape[0]
        return ll.to(W.dtype).reshape(())

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        gW, gV, gD, gmean, gspread, idx = ctx.saved_tensors
        return (None, None, g * gW, g * _scatter_gV(ctx.nV, gV, idx), g * gD, g * gmean, g * gspread, None, None, None, None,
                None)


def _scatter_gV(nV, gV, idx):
    """d/dV of the resident V from the minibatch's d/dV[idx] (a spot listed twice gets both contributions)."""
    if idx is None:
        return gV
    full = torch.zeros(nV, dtype=gV.dtype, device=gV.device)
    full.index_add_(0, idx, gV)
    return full


def _k7_dense(y, idx, W, V, D, mean, spread, eps, n_var, clamp_min, w_softplus, with_lgamma):
    """K7 on a dense G x N count matrix: gpz_poisson_fwdbwd_* (D None) or gpz_negbin_fwdbwd_* (D the raw dispersion).
    Returns gW, gV (minibatch), gmean, gspread, ll (one double), idx (int64 on the device or None) and gD (None for Poisson)."""
    dt = W.dtype
    G, F = W.shape
    # y: the reference passes floats; integer counts (uint8 / int16 / int32) are read as stored by the fp32 tensor-core kernel
    # (F <= 16), any other combination is converted on the device
    y_kind = PoissonLL.Y_KINDS.get(y.dtype, 0) if (dt == torch.float32 and F <= 16) else 0
    if y_kind == 0 and y.dtype != dt:
        y = y.to(dt)
    y = _c(y)
    B = mean.shape[1]
    E = eps.shape[0]
    assert y.shape[0] == G and mean.shape[0] == F and eps.shape[1] == F and eps.shape[2] == B
    if idx is not None:
        idx = _c(idx.to(device=W.device, dtype=torch.int64))
    else:
        assert y.shape[1] == B
    lib = _cabi.lib()
    suf = "f32" if dt == torch.float32 else "f64"
    name = "poisson" if D is None else "negbin"
    ws_bytes = int(getattr(lib, f"gpz_{name}_workspace_bytes_{suf}")(G, F, B, E))
    ws = torch.empty(ws_bytes // 8 + 1, dtype=torch.float64, device=W.device)
    ll = torch.empty(1, dtype=torch.float64, device=W.device)
    gW = torch.empty_like(W)
    gV = torch.empty(B, dtype=dt, device=W.device)
    gD = None if D is None else torch.empty_like(D)
    gmean = torch.empty_like(mean)
    gspread = torch.empty_like(spread)
    nb_in, nb_out = ((), ()) if D is None else ((D,), (gD,))
    tail = (y.shape[1], idx, W, int(w_softplus), V, *nb_in, mean, spread, eps, G, F, B, E, int(n_var), clamp_min,
            int(with_lgamma), ll, gW, gV, *nb_out, gmean, gspread, ws, ws_bytes)
    if y_kind:
        call(f"{name}_fwdbwd_yt", dt, y, y_kind, *tail)
    else:
        call(f"{name}_fwdbwd", dt, y, *tail)
    return gW, gV, gmean, gspread, ll, idx, gD


class GaussianLL(Function):
    """sum_{g,n} E_q[log N(y_gn | bias_g + sum_f W_gf F_fn, softplus(noise_g)^2)] under q(F) = N(mean, v), in closed form (no
    samples), with the gradients w.r.t. W, bias, noise, mean and spread from the same pass over y (K7-G, csrc/gaussian.cu).
    spread[f] is a variance (v = clamp(spread, clamp_min)) for f < n_var and a std-dev (v = spread^2) otherwise.
    y: dense G x N of any float or integer dtype (converted on the device to the compute dtype); idx: optional minibatch
    indices, y is read as y[:, idx]."""

    @staticmethod
    def forward(ctx, y, idx, W, bias, noise, mean, spread, n_var, clamp_min):
        if isinstance(y, SparseCounts):
            raise NotImplementedError(
                "the Gaussian likelihood has no sparse kernel yet: y enters only linearly and through sum y^2, so a sparse path "
                "is possible, but it is not built; pass y.to_dense()")
        W, bias, noise, mean, spread = _c(W), _c(bias), _c(noise), _c(mean), _c(spread)
        dt = W.dtype
        G, F = W.shape
        B = mean.shape[1]
        y = _c(y if y.dtype == dt else y.to(dt))
        assert y.shape[0] == G and mean.shape[0] == F and spread.shape == mean.shape
        assert bias.shape == (G,) and noise.shape == (G,) and bias.dtype == dt and noise.dtype == dt
        if idx is not None:
            idx = _c(idx.to(device=W.device, dtype=torch.int64))
        else:
            assert y.shape[1] == B
        suf = "f32" if dt == torch.float32 else "f64"
        ws_bytes = int(getattr(_cabi.lib(), "gpz_gaussian_workspace_bytes_" + suf)(G, F, B))
        ws = torch.empty(ws_bytes // 8 + 1, dtype=torch.float64, device=W.device)
        ll = torch.empty(1, dtype=torch.float64, device=W.device)
        gW, gbias, gnoise = torch.empty_like(W), torch.empty_like(bias), torch.empty_like(noise)
        gmean, gspread = torch.empty_like(mean), torch.empty_like(spread)
        call("gaussian_fwdbwd", dt, y, y.shape[1], idx, W, bias, noise, mean, spread, G, F, B, int(n_var), clamp_min, ll, gW, gbias,
             gnoise, gmean, gspread, ws, ws_bytes)
        ctx.save_for_backward(gW, gbias, gnoise, gmean, gspread)
        return ll.to(dt).reshape(())

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        gW, gbias, gnoise, gmean, gspread = ctx.saved_tensors
        return None, None, g * gW, g * gbias, g * gnoise, g * gmean, g * gspread, None, None


_CSC_KINDS = {torch.uint8: 1, torch.int16: 2, torch.int32: 3}      # count_kind of gpz_poisson_fwdbwd_csc_* (0 = the compute type)


def _poisson_csc(y, idx, W, V, mean, spread, eps, n_var, clamp_min, w_softplus, with_lgamma):
    """K7 on sparse counts: gpz_poisson_fwdbwd_csc_*.  Same outputs as the dense call."""
    dt = W.dtype
    G, F = W.shape
    B, E = mean.shape[1], eps.shape[0]
    N = y.shape[1]
    assert y.shape[0] == G and mean.shape[0] == F and eps.shape[1] == F and eps.shape[2] == B
    if idx is not None:
        idx = _c(idx.to(device=W.device, dtype=torch.int64))
    else:
        assert N == B
    vals = y.values
    kind = _CSC_KINDS.get(vals.dtype, 0)
    if kind == 0 and vals.dtype != dt:
        vals = vals.to(dt)
    suf = "f32" if dt == torch.float32 else "f64"
    ws_bytes = int(getattr(_cabi.lib(), "gpz_poisson_csc_workspace_bytes_" + suf)(G, F, B, E))
    ws = torch.empty(ws_bytes // 8 + 1, dtype=torch.float64, device=W.device)
    ll = torch.empty(1, dtype=torch.float64, device=W.device)
    gW, gV = torch.empty_like(W), torch.empty(B, dtype=dt, device=W.device)
    gmean, gspread = torch.empty_like(mean), torch.empty_like(spread)
    call("poisson_fwdbwd_csc", dt, y.indptr, y.genes, _c(vals), kind, N, idx, W, int(w_softplus), V, mean, spread, eps, G, F, B,
         E, int(n_var), clamp_min, int(with_lgamma), ll, gW, gV, gmean, gspread, ws, ws_bytes)
    return gW, gV, gmean, gspread, ll, idx


def poisson_rate(W, V, idx, F, w_softplus=True):
    """Materialised Poisson rate E x G x B (compatibility path, likelihoods.py:83-85); differentiable
    through `_PoissonRate`."""
    return _PoissonRate.apply(W, V, idx, F, w_softplus)


class _PoissonRate(Function):
    @staticmethod
    def forward(ctx, W, V, idx, F, w_softplus):
        W, V, F = _c(W), _c(V), _c(F)
        dt = W.dtype
        G, nF = W.shape
        E, _, B = F.shape
        if idx is not None:
            idx = _c(idx.to(device=W.device, dtype=torch.int64))
        rate = torch.empty((E, G, B), dtype=dt, device=W.device)
        call("poisson_rate", dt, W, int(w_softplus), V, idx, F, rate, G, nF, B, E)
        ctx.save_for_backward(W, V, F, idx, rate)
        ctx.w_softplus = w_softplus
        return rate

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        # rate = spV[n] * sum_f w[g,f] ef[e,f,n]; the three contractions below are our own batched GEMM.
        W, V, F, idx, rate = ctx.saved_tensors
        g = _c(g)
        E, G, B = g.shape
        Vb = V if idx is None else V[idx]
        spV = torch.nn.functional.softplus(Vb)
        ef = torch.exp(F)                                              # E x nF x B
        w = torch.nn.functional.softplus(W) if ctx.w_softplus else W
        gz = g * spV                                                   # d/d(zr)
        gF = gemm(w.unsqueeze(0).expand(E, -1, -1).contiguous(), gz, ta=True) * ef
        gw = gemm(gz, ef, tb=True).sum(0)
        if ctx.w_softplus:
            gw = gw * torch.sigmoid(W)
        gVb = (g * rate).sum((0, 1)) / spV * torch.sigmoid(Vb)
        if idx is not None:
            gV = torch.zeros_like(V)
            gV.index_add_(0, idx, gVb)
        else:
            gV = gVb
        return gw, gV, None, gF, None
