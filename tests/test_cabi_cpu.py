"""CPU: the C-ABI library builds, loads and exports every symbol include/gpzoo_b200.h declares; the product
path refuses CPU tensors loudly (there is no fallback)."""
import os

import pytest
import torch


@pytest.fixture(scope="module")
def lib():
    from gpzoo_b200 import _cabi, build
    if not os.path.exists(_cabi.LIB_PATH):
        build.build()
    return _cabi.lib()


def test_exports_match_header(lib):
    from gpzoo_b200 import _cabi
    syms = _cabi.exported_symbols()
    assert len(syms) >= 30
    missing = [s for s in syms if not hasattr(lib, s)]
    assert not missing, missing
    assert lib.gpz_abi_version() >= 1
    assert b"success" in lib.gpz_error_string(0)


def test_every_prototype_binds(lib):
    """Each declared symbol gets the header's types: one argtype per parameter (counted here from the raw prototype text) and
    the C return type; every entry point that takes a stream takes it last, as `call()` appends it."""
    import ctypes
    import re
    from gpzoo_b200 import _cabi
    txt = open(_cabi.HEADER).read()
    special = {"gpz_error_string": ctypes.c_char_p, "gpz_launch_count": ctypes.c_longlong}
    for sym, proto in _cabi.prototypes().items():
        fn = getattr(lib, sym)
        plist = re.search(rf"\b{sym}\s*\(([^)]*)\)\s*;", txt).group(1).strip()
        n = 0 if plist == "void" else plist.count(",") + 1
        assert len(fn.argtypes) == n == len(proto.params), sym
        want = special.get(sym, ctypes.c_int64 if "_workspace_bytes_" in sym else ctypes.c_int)
        assert fn.restype is want, (sym, fn.restype)
        names = [p.name for p in proto.params]
        if "stream" in names:
            assert names.index("stream") == n - 1 and proto.params[-1].ctype == "void*", sym
    assert lib.gpz_error_string.argtypes == (ctypes.c_int,)
    assert len(lib.gpz_umma_gemm_f32.argtypes) == 25 and len(lib.gpz_adam_step_f64.argtypes) == 13


def test_header_parser_rejects_unknown_types():
    from gpzoo_b200 import _cabi
    ok = _cabi.parse_header("/* c */\n#define X 1\nlong long gpz_a(void);\nint gpz_b_f32(void* const* t, const int64_t* n, "
                            "double x, void* stream);")
    assert set(ok) == {"gpz_a", "gpz_b_f32"} and ok["gpz_a"].params == ()
    assert [(p.name, p.ctype) for p in ok["gpz_b_f32"].params] == [("t", "void**"), ("n", "int64_t*"), ("x", "double"),
                                                                    ("stream", "void*")]
    with pytest.raises(_cabi.GpzError, match=r"half\*.*gpz_c_f32"):
        _cabi.parse_header("int gpz_c_f32(const half* x, int n, void* stream);")
    with pytest.raises(_cabi.GpzError, match=r"unsigned.*gpz_d"):
        _cabi.parse_header("unsigned gpz_d(void);")


@pytest.fixture
def no_stream(monkeypatch):
    """`call()` without a CUDA stream.  Every call below fails a check before the library is entered; its sizes are all 0, so
    even a call that got through would launch nothing and touch no memory."""
    from gpzoo_b200 import _cabi
    monkeypatch.setattr(_cabi, "stream", lambda: None)


def test_call_checks_argument_count(lib, no_stream):
    from gpzoo_b200 import _cabi
    # gpz_tri_op_f32(const float* in, float* out, int M, int L, int mode, void* stream)
    with pytest.raises(_cabi.GpzError, match=r"gpz_tri_op_f32 takes 5 arguments before the stream, got 6"):
        _cabi.call("tri_op", torch.float32, None, None, 0, 0, 0, 0)
    with pytest.raises(_cabi.GpzError, match=r"gpz_tri_op_f32 takes 5 arguments before the stream, got 4"):
        _cabi.call("tri_op", torch.float32, None, None, 0, 0)


def test_call_checks_argument_types(lib, no_stream):
    from gpzoo_b200 import _cabi
    f64 = torch.zeros(4, dtype=torch.float64)
    with pytest.raises(_cabi.GpzError, match=r"gpz_tri_op_f32: parameter in is float\*, got a torch.float64 tensor"):
        _cabi.call("tri_op", torch.float32, f64, None, 0, 0, 0)
    with pytest.raises(_cabi.GpzError, match=r"gpz_tri_op_f64: parameter out is double\*, got a torch.float32 tensor"):
        _cabi.call("tri_op", torch.float64, None, f64.float(), 0, 0, 0)
    with pytest.raises(_cabi.GpzError, match=r"gpz_chol_inv_f32: parameter info is int\*, got a torch.int64 tensor"):
        _cabi.call("chol_inv", torch.float32, None, None, None, None, 0, 0, torch.zeros(1, dtype=torch.int64))
    # void* takes any dtype: these get past the dtype check and stop at the CUDA check
    for dt in (torch.float16, torch.uint8, torch.int16, torch.float64):
        with pytest.raises(_cabi.GpzError, match="need CUDA tensors"):
            _cabi.call("split16", torch.float32, None, 0, 0, 0, torch.zeros(4, dtype=dt), None, None, None, None, None)
    with pytest.raises(_cabi.GpzError, match="need CUDA tensors"):
        _cabi.call("tri_op", torch.float32, f64.float(), None, 0, 0, 0)
    with pytest.raises(_cabi.GpzError, match=r"gpz_tri_op_f32: parameter M \(int\)"):
        _cabi.call("tri_op", torch.float32, None, None, 0.0, 0, 0)
    with pytest.raises(_cabi.GpzError, match=r"gpz_tri_op_f32: parameter M is int, got a tensor"):
        _cabi.call("tri_op", torch.float32, None, None, torch.zeros(()), 0, 0)
    with pytest.raises(_cabi.GpzError, match=r"gpz_tri_op_f32: parameter in is float\*, got int"):
        _cabi.call("tri_op", torch.float32, 0, None, 0, 0, 0)


def test_literal_call_sites_match_the_header():
    """Every `call("<literal>", dtype, ...)` in the package names a declared entry point, with one argument per parameter before
    the stream wherever the arguments are written out."""
    import ast
    import glob
    from gpzoo_b200 import _cabi
    protos = _cabi.prototypes()
    root = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpzoo_b200")
    seen = 0
    for path in glob.glob(os.path.join(root, "*.py")):
        for node in ast.walk(ast.parse(open(path).read())):
            if not (isinstance(node, ast.Call) and getattr(node.func, "id", getattr(node.func, "attr", None)) == "call"
                    and node.args and isinstance(node.args[0], ast.Constant)):
                continue
            seen += 1
            where = f"{os.path.basename(path)}:{node.lineno}"
            syms = [f"gpz_{node.args[0].value}_{s}" for s in ("f32", "f64") if f"gpz_{node.args[0].value}_{s}" in protos]
            assert syms, where
            if not any(isinstance(a, ast.Starred) for a in node.args):
                for s in syms:
                    assert len(node.args) - 2 == len(protos[s].params) - 1, (where, s)
    assert seen >= 30


def test_no_cpu_fallback(lib):
    import gpzoo_b200 as gz
    k = gz.kernels.NSF_RBF(L=2)
    with pytest.raises(gz._cabi.GpzError):
        k(torch.randn(5, 2), torch.randn(3, 2))


def test_initialisation_has_no_host_path():
    """The initialisation pipeline (SURVEY 8(f) row 4) refuses to run without a CUDA device; its pure formulas need none."""
    import numpy as np
    from gpzoo_b200 import initialisation as I, utilities as U
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            I.nmf(np.ones((6, 4)), 2)
        with pytest.raises(RuntimeError):
            U.regularized_nmf(np.ones((6, 4)), 2)
    mu, sd = U.lnormal_approx_dirichlet(4)
    assert abs(mu - (-np.log(4) - (np.log(8) - np.log(5)) / 2)) < 1e-15 and abs(sd - np.sqrt(np.log(8) - np.log(5))) < 1e-15
    assert set(("regularized_nmf", "shrink_factors", "shrink_loadings", "init_softplus", "rescale_spatial_coords",
                "build_group_distances", "lnormal_approx_dirichlet")) <= set(dir(U))


def test_product_never_imports_oracle():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for dirpath, _, files in os.walk(os.path.join(root, "gpzoo_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


def test_fused_adam_and_tiled_predict_refuse_cpu(lib):
    """The pieces next to the path have no CPU route either: the fused optimiser and the tiled predictor raise on CPU tensors."""
    import gpzoo_b200 as gz
    p = torch.nn.Parameter(torch.randn(7))
    p.grad = torch.randn(7)
    with pytest.raises(gz._cabi.GpzError):
        gz.optim.Adam([p], lr=1e-2).step()
    gp = gz.gp.SVGP(gz.kernels.NSF_RBF(L=2), dim=2, M=8, jitter=1e-2)
    gp.mu = torch.nn.Parameter(torch.zeros(2, 8))
    gp.Lu = torch.nn.Parameter(torch.eye(8).expand(2, -1, -1).contiguous())
    with pytest.raises(gz._cabi.GpzError):
        gp.predict_moments(torch.randn(20, 2), tile=8)


def test_abi_version_and_new_entry_points(lib):
    """ABI 2 added `kind` to the kernel-build calls; the split-FP16 / large-M / training-step entry points are exported."""
    assert lib.gpz_abi_version() >= 2
    for s in ("gpz_kernel_build_fwd_h_f32", "gpz_svgp_predict_fwd_h_f32", "gpz_svgp_predict_bwd_h_f32", "gpz_split16_f32",
              "gpz_umma_gemm16_f32", "gpz_chol_inv_tc_f32", "gpz_adam_step_f32", "gpz_adam_step_f64", "gpz_svgp_predict_h_stat_row"):
        assert hasattr(lib, s), s
    assert lib.gpz_svgp_predict_h_supported(1024, 32768) == 1 and lib.gpz_svgp_predict_h_supported(1020, 32768) == 0
    rows = [lib.gpz_svgp_predict_h_stat_row(i) for i in range(5)]
    assert len(set(rows)) == 5 and min(rows) >= 0                       # five distinct rows of the stats block
    assert lib.gpz_svgp_predict_h_stat_row(99) == -1


def test_state_dict_keys_and_shapes_match_reference():
    """Every model family has the reference's state_dict keys and shapes (golden written from the unmodified reference by
    oracle/gen_golden.py; compared live as well when /root/reference is present).  Module construction needs no GPU."""
    import json
    import os
    import types
    import gpzoo_b200 as gz
    from oracle import ref_loader, ref_runner
    from tests.helpers import GOLDEN
    golden = json.load(open(os.path.join(GOLDEN, "state_dict_shapes.json")))
    ours = ref_runner.state_dict_shapes(types.SimpleNamespace(kernels=gz.kernels, gp=gz.gp, likelihoods=gz.likelihoods))
    assert set(ours) == set(golden)
    for name in golden:
        assert ours[name] == golden[name], (name, ours[name], golden[name])
    if ref_loader.available():
        assert ref_runner.state_dict_shapes() == golden


def test_reference_utility_names_importable():
    """`from gpzoo.utilities import ...` of every hot-path name keeps working after install_as_gpzoo() (SURVEY.md §2.1 row 11)."""
    import sys
    import gpzoo_b200 as gz
    saved = {k: v for k, v in sys.modules.items() if k == "gpzoo" or k.startswith("gpzoo.")}
    gz.install_as_gpzoo()
    try:
        _check_reference_names()
    finally:                                  # other tests import the real reference under the same name
        for k in [k for k in sys.modules if k == "gpzoo" or k.startswith("gpzoo.")]:
            del sys.modules[k]
        sys.modules.update(saved)


def _check_reference_names():
    from gpzoo.utilities import (_embed_distance_matrix, _squared_dist, _torch_sqrt, add_jitter, reshape_param, svgp_forward,  # noqa: F401
                                 train, train_batched, train_closure_batched, train_hybrid, train_hybrid_batched, whitened_KL)
    from gpzoo.gp import MGGP_WSVGP, WSVGP
    from gpzoo.likelihoods import Hybrid_NSF2
    assert hasattr(WSVGP, "forward_precomputed") and hasattr(MGGP_WSVGP, "forward_precomputed")
    assert hasattr(Hybrid_NSF2, "forward_precomputed")
    import torch
    assert reshape_param(torch.zeros(2, 3, 4, 5)).shape == (6, 4, 5)
    assert abs(float(_torch_sqrt(torch.zeros((), dtype=torch.float64), 1e-6)) - 1e-3) < 1e-15
