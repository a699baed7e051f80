"""The dense fused Poisson ELBO (K7, gpz_poisson_fwdbwd_* in csrc/poisson.cu) against a float64 autograd reference on the device,
at the grid shapes the benchmark runs: gene ranges of several 16-gene blocks and several gene chunks per CTA, ragged chunks and
ranges, a single range, every factor-count template, narrow integer counts, data drawn near a fit, and layout and value edges.

Near a fit t = (y / r - 1) / E cancels across spots, so each output is checked as ||out - ref|| <= c ||mag||, where mag is the same
reference sum taken over the absolute values of its summands.  A dropped or double-counted 16-gene block moves an output by about
||mag|| / (blocks per range), orders above either c.  The CPU test checks, through a mirror of poisson_grid, that the shape table
reaches every kind of gene-range split of both kernels."""
import time

import pytest
import torch
import torch.nn.functional as Fnn

from tests.helpers import relerr

DEV = "cuda"
OUTS = ("ll", "W", "V", "mean", "spread")

# fp64: exact log and division, 1e-11 of the magnitude.
C64, REL64 = 1e-11, 1e-11
# fp32.  poisson_kernel4 (F <= 16) splits every operand x into bf16 hi + lo with |x - hi - lo| <= 2^-18 |x| and forms a product as
# hi*hi + hi*lo + lo*hi, dropping lo*lo (<= 2^-18 |ab|): each product term is within 3 * 2^-18 = 1.1e-5 of exact.  The rate carries
# that error into y / r, hence into t, whose magnitude term is (y / r + 1) / E; the second contraction (t with w into d/dF, t with EF'
# into d/dW) adds its own 1.1e-5: 2.3e-5 of ||mag|| to first order.  The fp32 sums behind it (MMA accumulation, the D3 exchange over
# 8 warps, the gW partials of at most 1185 CTAs, the D2 atomics over the gene ranges) are bounded by n 2^-24 for n terms but, rounded
# to nearest, grow as sqrt(n) 2^-24 (< 3e-6 for every shape here).  poisson_kernel2 (F > 16) is plain fp32 FMA with __logf (2^-21
# absolute) and __fdividef (2 ulp): its contractions are within F 2^-24 and its sums within (genes per CTA + spots per CTA /
# 64 + CTAs) 2^-24 = 1.5e-5 at worst.  Both stay within 3e-5.
C32, REL32 = 3e-5, 3e-5


# ---- grid mirror ------------------------------------------------------------------------------------------------------------
def _cdiv(a, b):
    return -(-a // b)


def poisson_grid(G, F, B, is_f32):
    """Mirror of poisson_grid in gpzoo_b200/csrc/poisson.cu: (path, nbx, nby, gpc) of the dense K7 launch.  Path "tc" is
    poisson_kernel4 (fp32, F <= 16: 256 spots per CTA, gene ranges in whole 16-gene blocks staged as 64-gene chunks), path "k2"
    poisson_kernel2 (fp64, and fp32 with F > 16: 256 spots per CTA, gene ranges in 32-gene chunks)."""
    nbx = _cdiv(B, 256)
    if is_f32 and F <= 16:
        blocks = _cdiv(G, 16)
        by = min(blocks, max(1, 1184 // nbx)) if nbx < 1184 else 1
        gpc = 16 * _cdiv(blocks, by)
        return "tc", nbx, _cdiv(G, gpc), gpc
    chunks = _cdiv(G, 32)
    by = min(chunks, _cdiv(1184, nbx)) if nbx < 1184 else 1
    gpc = 32 * _cdiv(chunks, by)
    return "k2", nbx, _cdiv(G, gpc), gpc


def _workspace_bytes(G, F, B, E, is_f32):
    """Mirror of poisson_ws_bytes in csrc/poisson.cu: it depends on the grid, so the library's answer checks poisson_grid above."""
    path, nbx, nby, _ = poisson_grid(G, F, B, is_f32)
    b = 8 * ((nbx * nby + 3) & ~1) + _cdiv((4 if is_f32 else 8) * nbx * G * F, 16) * 16
    if path == "tc":
        eb16 = 16 * E * B
        b += 4 * 16 * G + 4 * eb16 + 4 * eb16 + 4 * 16 * nby + 8 * _cdiv(B, 64) + 16
    return b


def _categories(path, G, gpc, nby, E, has_idx):
    """The kinds of gene-range split a launch exercises (chunk: 64 genes on "tc", 32 on "k2")."""
    chunk = 64 if path == "tc" else 32
    last = G - (nby - 1) * gpc                                  # genes of the last range
    c = set()
    if gpc == (16 if path == "tc" else 32):
        c.add("one_unit")                                       # one 16-gene block (tc) / one chunk (k2) per range: the control
    if path == "tc" and 16 < gpc <= 64:
        c.add("blocks_in_chunk")                                # jb >= 1 inside one chunk
    if gpc == 64:
        c.add("full_chunk" if path == "tc" else "two_chunks")
    if gpc > chunk and (gpc % chunk or last % chunk):
        c.add("chunk_and_ragged_chunk")
    if gpc > 2 * chunk and G % gpc:
        c.add("chunks_and_ragged_range")
    if nby == 1:
        c.add("single_range")
    if E > 1 and gpc > chunk // (4 if path == "tc" else 1):
        c.add("samples_over_multi_unit_range")                  # the y prefetch wraps to the next sample across blocks / chunks
    if has_idx and gpc > chunk // (4 if path == "tc" else 1):
        c.add("idx_multi_unit_range")
    return c


REQUIRED = {
    "tc": {"one_unit", "blocks_in_chunk", "full_chunk", "chunk_and_ragged_chunk", "chunks_and_ragged_range", "single_range",
           "samples_over_multi_unit_range", "idx_multi_unit_range"},
    "k2": {"one_unit", "two_chunks", "chunk_and_ragged_chunk", "chunks_and_ragged_range", "single_range",
           "samples_over_multi_unit_range", "idx_multi_unit_range"},
}

# name: G, Ntot (resident spots), B (minibatch through idx; None: all spots), E, and the (nbx, nby, gpc) of each path at F = 10
SHAPES = {
    "g16": dict(G=2000, Ntot=1024, B=None, E=1, tc=(4, 125, 16), k2=(4, 63, 32)),              # every existing test's split
    "cfg3_E10": dict(G=2000, Ntot=4000, B=None, E=10, tc=(16, 63, 32), k2=(16, 63, 32)),
    "cfg4_idx": dict(G=2000, Ntot=12500, B=8192, E=1, tc=(32, 32, 64), k2=(32, 32, 64)),
    "ragged_chunk": dict(G=1000, Ntot=20000, B=None, E=1, tc=(79, 13, 80), k2=(79, 11, 96)),
    "cfg2": dict(G=2000, Ntot=32768, B=None, E=1, tc=(128, 9, 224), k2=(128, 9, 224)),
    "single_range": dict(G=40, Ntot=303360, B=None, E=2, tc=(1185, 1, 48), k2=(1185, 1, 64)),
    "odd_B": dict(G=1000, Ntot=20001, B=None, E=1, tc=(79, 13, 80), k2=(79, 11, 96)),
    "idx_dup": dict(G=1000, Ntot=25000, B=20000, E=2, tc=(79, 13, 80), k2=(79, 11, 96)),
}
FP64_FACTORS = (1, 4, 5, 12, 13, 20, 21, 32)                   # across every FMAX boundary of poisson_kernel2 (4, 12, 20, 32)
FP32_FACTORS = (1, 16, 17, 32)                                 # tensor-core path up to 16, then poisson_kernel2 (FMAX 20, 32)


def test_shape_table_covers_every_split_and_workspace_size():
    """CPU: the table's labels are what poisson_grid gives, the library agrees, and every kind of split is reached on both paths."""
    import os
    from gpzoo_b200 import _cabi, build
    if not os.path.exists(_cabi.LIB_PATH):
        build.build()
    lib = _cabi.lib()
    seen = {"tc": set(), "k2": set()}
    for name, s in SHAPES.items():
        B = s["B"] or s["Ntot"]
        for path, is_f32 in (("tc", True), ("k2", False)):
            p, nbx, nby, gpc = poisson_grid(s["G"], 10, B, is_f32)
            assert p == path and (nbx, nby, gpc) == s[path], (name, path, (nbx, nby, gpc))
            seen[path] |= _categories(path, s["G"], gpc, nby, s["E"], s["B"] is not None)
    for F in FP32_FACTORS + FP64_FACTORS:                         # every factor count runs at the ragged-chunk shape
        for is_f32 in (True, False):
            p, nbx, nby, gpc = poisson_grid(1000, F, 20000, is_f32)
            assert (nbx, nby, gpc) == SHAPES["ragged_chunk"][p]
    assert seen["tc"] >= REQUIRED["tc"], REQUIRED["tc"] - seen["tc"]
    assert seen["k2"] >= REQUIRED["k2"], REQUIRED["k2"] - seen["k2"]
    for s in SHAPES.values():
        for F in (1, 10, 16, 17, 32):
            for is_f32, suf in ((True, "f32"), (False, "f64")):
                args = (s["G"], F, s["B"] or s["Ntot"], s["E"])
                got = getattr(lib, "gpz_poisson_workspace_bytes_" + suf)(*args)
                assert got == _workspace_bytes(*args, is_f32), (args, suf)


# ---- inputs, kernel, reference ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module", autouse=True)
def _report():
    """Prints the module's wall time and peak device memory (run with -s to see it)."""
    t0 = time.perf_counter()
    if torch.cuda.is_available():
        torch.cuda.reset_peak_memory_stats()
    yield
    if torch.cuda.is_available():
        print(f"\n[poisson shapes] {time.perf_counter() - t0:.1f} s, peak max_memory_allocated "
              f"{torch.cuda.max_memory_allocated() / 2**30:.2f} GiB")


def _problem(G, Ntot, B, E, dt, F=10, seed=0, near=False, soft=True):
    """Seeded inputs on the device, rounded to dt so the reference sees what the kernel sees.  Far from a fit: y ~ Poisson(U(0, 2))
    against rates ~ 10.  Near a fit: softplus(W) ~ 0.05-0.13 (rates ~ 1) and y ~ Poisson(reference rate)."""
    from oracle import gpzoo_oracle as O
    g = torch.Generator(device=DEV).manual_seed(seed)
    rand = lambda *s: torch.rand(*s, generator=g, device=DEV, dtype=torch.float64)
    randn = lambda *s: torch.randn(*s, generator=g, device=DEV, dtype=torch.float64)
    idx = None if B is None else torch.randperm(Ntot, generator=g, device=DEV)[:B]
    B = Ntot if B is None else B
    p = dict(idx=idx, W=rand(G, F) - (3.0 if near else 0.0) + (0.0 if soft else 0.1), V=1 + 0.2 * randn(Ntot),
             mean=0.3 * randn(F, B), spread=0.05 + 0.3 * rand(F, B), eps=randn(E, F, B), nvar=(F + 1) // 2,
             cm=float(torch.tensor(5e-2, dtype=dt)), soft=soft, E=E)
    p["spread"][0, :7] = 1e-3                                  # below the variance clamp
    for k in ("W", "V", "mean", "spread", "eps"):
        p[k] = p[k].to(dt).double()
    if near:
        assert idx is None
        rate = O.poisson_rate(p["W"], p["mean"] + p["eps"] * _sd(p, p["spread"]), p["V"], softplus_W=soft).mean(0)
        p["y"] = torch.poisson(rate, generator=g)
    else:
        p["y"] = torch.poisson(2 * rand(G, Ntot), generator=g)
    return p


def _sd(p, spread):
    nv = p["nvar"]
    return torch.cat((spread[:nv].clamp(min=p["cm"]).sqrt(), spread[nv:]), 0)


def _kernel(p, y, dt, with_lgamma=True, entry="poisson_fwdbwd"):
    """PoissonLL on the device: ll and the gradients w.r.t. W, V, mean, spread (dV scattered through idx by PoissonLL.backward)."""
    from gpzoo_b200 import _cabi, functional as F
    lv = [p[k].to(dt).requires_grad_(True) for k in ("W", "V", "mean", "spread")]
    _cabi.profile = {}
    try:
        out = F.PoissonLL.apply(y, p["idx"], *lv, p["eps"].to(dt), p["nvar"], p["cm"], p["soft"], with_lgamma)
    finally:
        calls, _cabi.profile = set(_cabi.profile), None
    assert entry in calls, calls
    out.backward()
    return [out.detach()] + [t.grad for t in lv]


def _reference(p, with_lgamma=True, y=None):
    """float64 autograd through oracle.poisson_rate / poisson_loglik (plain torch ops on the device), and for each output the
    magnitude: the same sum over the absolute values of its summands, in closed form."""
    from oracle import gpzoo_oracle as O
    y = p["y"] if y is None else y
    idx, eps, soft, E, nv = p["idx"], p["eps"], p["soft"], p["E"], p["nvar"]
    leaves = [p[k].clone().requires_grad_(True) for k in ("W", "V", "mean", "spread")]
    Wl, Vl, ml, sl = leaves
    rate = O.poisson_rate(Wl, ml + eps * _sd(p, sl), Vl if idx is None else Vl[idx], softplus_W=soft)
    yb = (y if idx is None else y[:, idx]).double()
    ll = O.poisson_loglik(yb, rate, with_lgamma=with_lgamma)
    ref = [ll.detach()] + list(torch.autograd.grad(ll, leaves))
    del ll
    with torch.no_grad():
        r = rate.detach()
        del rate
        W, V, spread = p["W"], p["V"], p["spread"]
        Vb = V if idx is None else V[idx]
        spV = Fnn.softplus(Vb)
        sd = _sd(p, spread)
        ef = spV * torch.exp(p["mean"] + eps * sd)                      # EF' = softplus(V) exp(F): E x F x B
        w = (Fnn.softplus(W) if soft else W).abs()
        dw = torch.sigmoid(W) if soft else torch.ones_like(W)
        a = (yb / r + 1) / E                                           # >= |t|, t = d ll / d rate' = (y / r - 1) / E
        m_ll = ((torch.xlogy(yb, r).abs() + r) / E).sum() + (torch.lgamma(yb + 1).abs().sum() if with_lgamma else 0.0)
        m_W = torch.matmul(a, ef.transpose(1, 2)).sum(0) * dw
        u = torch.matmul(w.t(), a)                                     # sum_g (y / r + 1) / E |w[g, f]|: E x F x B
        m_mean = (ef * u).sum(0)
        m_spread = (ef * eps.abs() * u).sum(0)
        m_spread[:nv] *= torch.where(spread[:nv] >= p["cm"], 1 / (2 * sd[:nv]), torch.zeros_like(sd[:nv]))
        m_Vb = torch.sigmoid(Vb) / spV * ((yb + r) / E).sum((0, 1))
        m_V = m_Vb if idx is None else torch.zeros_like(V).index_add_(0, idx, m_Vb)
        del r, a, u
    return ref, [m_ll, m_W, m_V, m_mean, m_spread]


def _check(label, out, ref, mag, c, rel=None):
    """||out - ref|| <= c ||mag|| for every output; with rel, also the plain relative error (far from a fit)."""
    scaled = {k: (o.double() - r).norm().item() / m.norm().item() for k, o, r, m in zip(OUTS, out, ref, mag)}
    worst = max(scaled, key=scaled.get)
    msg = f"{label}: max ||out-ref||/||mag|| = {scaled[worst]:.2e} ({worst})"
    if rel is not None:
        rels = {k: relerr(o, r) for k, o, r in zip(OUTS, out, ref)}
        wr = max(rels, key=rels.get)
        msg += f", max relerr = {rels[wr]:.2e} ({wr})"
    print("\n" + msg)
    assert all(v <= c for v in scaled.values()), (label, scaled)
    if rel is not None:
        assert all(v < rel for v in rels.values()), (label, rels)


def _tols(dt):
    return (C64, REL64) if dt == torch.float64 else (C32, REL32)


DTS = [torch.float32, torch.float64]


# ---- gene-range splits ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTS, ids=["f32", "f64"])
@pytest.mark.parametrize("case", ["g16", "cfg3_E10", "cfg4_idx", "ragged_chunk", "cfg2", "cfg2_near", "single_range"])
def test_gene_range_splits(case, dt):
    near = case.endswith("_near")
    s = SHAPES[case[:-5] if near else case]
    p = _problem(s["G"], s["Ntot"], s["B"], s["E"], dt, seed=1, near=near)
    out = _kernel(p, p["y"].to(dt), dt)
    ref, mag = _reference(p)
    c, rel = _tols(dt)
    _check(f"{case} {dt}", out, ref, mag, c, None if near else rel)


@pytest.mark.gpu
@pytest.mark.parametrize("dt,F", [(torch.float32, f) for f in FP32_FACTORS] + [(torch.float64, f) for f in FP64_FACTORS],
                         ids=[f"f32-F{f}" for f in FP32_FACTORS] + [f"f64-F{f}" for f in FP64_FACTORS])
def test_factor_counts(dt, F):
    s = SHAPES["ragged_chunk"]
    p = _problem(s["G"], s["Ntot"], s["B"], s["E"], dt, F=F, seed=2)
    out = _kernel(p, p["y"].to(dt), dt)
    ref, mag = _reference(p)
    c, rel = _tols(dt)
    _check(f"F={F} {dt}", out, ref, mag, c, rel)


# ---- counts and inputs at config 2's shape, fp32 ---------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["uint8", "int16", "int32", "float_nonint", "no_lgamma"])
def test_counts_cfg2_fp32(kind):
    s = SHAPES["cfg2"]
    dt = torch.float32
    p = _problem(s["G"], s["Ntot"], s["B"], s["E"], dt, seed=3)
    g = torch.Generator(device=DEV).manual_seed(4)
    y = p["y"]
    entry = "poisson_fwdbwd"
    if kind in ("uint8", "int16", "int32"):
        top = 256 if kind == "uint8" else 4000                      # counts >= 64 take lfact_slow
        big = torch.rand(y.shape, generator=g, device=DEV) < 0.01
        y = torch.where(big, torch.randint(64, top, y.shape, generator=g, device=DEV, dtype=torch.float64), y)
        p["y"] = y
        y = y.to(getattr(torch, kind))
        entry = "poisson_fwdbwd_yt"
    elif kind == "float_nonint":
        y = p["y"] = 3 * torch.rand(y.shape, generator=g, device=DEV, dtype=torch.float64).to(dt).double()
    with_lgamma = kind != "no_lgamma"
    out = _kernel(p, y.to(dt) if y.is_floating_point() else y, dt, with_lgamma=with_lgamma, entry=entry)
    ref, mag = _reference(p, with_lgamma=with_lgamma)
    _check(f"cfg2 {kind}", out, ref, mag, C32, REL32)


# ---- memory layout ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTS, ids=["f32", "f64"])
def test_odd_row_length(dt):
    """B odd with no idx: y_ld is odd, so the tensor-core kernel cannot take its paired-column loads."""
    s = SHAPES["odd_B"]
    p = _problem(s["G"], s["Ntot"], s["B"], s["E"], dt, seed=5)
    out = _kernel(p, p["y"].to(dt), dt)
    ref, mag = _reference(p)
    c, rel = _tols(dt)
    _check(f"odd B {dt}", out, ref, mag, c, rel)


@pytest.mark.gpu
def test_uint8_counts_at_odd_address():
    """uint8 counts in a contiguous view whose base address is odd (one byte into its buffer)."""
    s = SHAPES["cfg2"]
    p = _problem(s["G"], s["Ntot"], s["B"], s["E"], torch.float32, seed=6)
    buf = torch.empty(s["G"] * s["Ntot"] + 1, dtype=torch.uint8, device=DEV)
    y = buf[1:].view(s["G"], s["Ntot"])
    y.copy_(p["y"].to(torch.uint8))
    assert y.is_contiguous() and y.data_ptr() % 2 == 1
    out = _kernel(p, y, torch.float32, entry="poisson_fwdbwd_yt")
    ref, mag = _reference(p)
    _check("uint8 at an odd address", out, ref, mag, C32, REL32)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTS, ids=["f32", "f64"])
def test_unsorted_idx_with_a_repeated_spot(dt):
    s = SHAPES["idx_dup"]
    p = _problem(s["G"], s["Ntot"], s["B"], s["E"], dt, seed=7)
    p["idx"][s["B"] - 3] = p["idx"][11]                        # one spot twice: its two dV contributions add up
    assert not bool((p["idx"][1:] >= p["idx"][:-1]).all())
    out = _kernel(p, p["y"].to(dt), dt)
    ref, mag = _reference(p)
    c, rel = _tols(dt)
    _check(f"idx with a repeat {dt}", out, ref, mag, c, rel)


# ---- values at the edges -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTS, ids=["f32", "f64"])
def test_softplus_threshold_and_clamp_equality(dt):
    """W and V at and above softplus's threshold of 20 (softplus(x) = x, gradient 1 above it), and variances exactly at clamp_min
    (torch's clamp passes the gradient at equality; the kernels test >=)."""
    s = SHAPES["ragged_chunk"]
    p = _problem(s["G"], s["Ntot"], s["B"], s["E"], dt, seed=8)
    p["W"][3, 2], p["W"][517, 4], p["W"][999, 9] = 20.0, 23.5, 20.0
    p["V"][5], p["V"][19999] = 20.0, 31.0
    p["spread"][0, 100:110] = p["cm"]
    p["spread"][p["nvar"] - 1, 5000:5003] = p["cm"]
    out = _kernel(p, p["y"].to(dt), dt)
    ref, mag = _reference(p)
    c, rel = _tols(dt)
    _check(f"softplus threshold / clamp equality {dt}", out, ref, mag, c, rel)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTS, ids=["f32", "f64"])
def test_raw_loadings_multi_chunk(dt):
    """w_softplus = False (Hybrid_NSF's raw, positive loadings) at the ragged-chunk shape."""
    s = SHAPES["ragged_chunk"]
    p = _problem(s["G"], s["Ntot"], s["B"], s["E"], dt, seed=9, soft=False)
    out = _kernel(p, p["y"].to(dt), dt)
    ref, mag = _reference(p)
    c, rel = _tols(dt)
    _check(f"raw loadings {dt}", out, ref, mag, c, rel)


# ---- compatibility path: the materialised rate --------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTS, ids=["f32", "f64"])
@pytest.mark.parametrize("with_idx", [False, True])
def test_rate_compat_vs_oracle(dt, with_idx):
    """functional.poisson_rate (gpz_poisson_rate_*) and its backward against oracle.poisson_rate: G not a multiple of the kernel's
    32-gene rows, E = 3."""
    from oracle import gpzoo_oracle as O
    from gpzoo_b200 import functional as F
    g = torch.Generator(device=DEV).manual_seed(10)
    G, Fn, Ntot, E = 77, 5, 300, 3
    idx = torch.randperm(Ntot, generator=g, device=DEV)[:170] if with_idx else None
    B = 170 if with_idx else Ntot
    W = torch.rand(G, Fn, generator=g, device=DEV, dtype=torch.float64).to(dt).double()
    V = (1 + 0.2 * torch.randn(Ntot, generator=g, device=DEV, dtype=torch.float64)).to(dt).double()
    Fs = (0.3 * torch.randn(E, Fn, B, generator=g, device=DEV, dtype=torch.float64)).to(dt).double()
    wt = torch.randn(E, G, B, generator=g, device=DEV, dtype=torch.float64)
    leaves = [t.clone().requires_grad_(True) for t in (W, V, Fs)]
    rate = O.poisson_rate(leaves[0], leaves[2], leaves[1] if idx is None else leaves[1][idx])
    (rate * wt).sum().backward()
    dl = [t.to(dt).requires_grad_(True) for t in (W, V, Fs)]
    out = F.poisson_rate(dl[0], dl[1], idx, dl[2], True)
    (out * wt.to(dt)).sum().backward()
    tol = REL64 if dt == torch.float64 else REL32
    assert out.shape == (E, G, B) and relerr(out, rate) < tol
    for name, a, b in zip(("W", "V", "F"), dl, leaves):
        assert relerr(a.grad, b.grad) < tol, (name, relerr(a.grad, b.grad))
