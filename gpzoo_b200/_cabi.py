"""ctypes binding of include/gpzoo_b200.h.

The CUDA shared library is the product: if it is missing or a call fails, this module raises — there is
no PyTorch / CPU fallback anywhere in the package.

The header is the only description of the C ABI: the argument and return types of every entry point are read from its
prototypes, and `call()` checks each call against them (argument count, the dtype of every tensor a pointer parameter
receives) on the host, before anything reaches the device.
"""
from __future__ import annotations

import ctypes
import os
import re
import threading
from typing import NamedTuple

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GPZ_LIB") or os.path.join(_HERE, "lib", "libgpzoo_b200.so")     # GPZ_LIB: A/B runs of two builds
HEADER = os.path.join(os.path.dirname(_HERE), "include", "gpzoo_b200.h")
_lib = None
_lock = threading.Lock()
launch_count = 0          # number of C-ABI compute calls issued (bench.py reports kernel launches from this)


class GpzError(RuntimeError):
    pass


# the C types the header uses, written without `const` and without a space before '*' ("void* const*" -> "void**")
_SCALARS = {"int": ctypes.c_int, "int64_t": ctypes.c_int64, "long long": ctypes.c_longlong, "float": ctypes.c_float,
            "double": ctypes.c_double}
_RESTYPES = {**_SCALARS, "char*": ctypes.c_char_p}
# pointer parameter -> dtype of the tensor it takes (None: any dtype; void** is a host array of device pointers)
_POINTERS = {"float*": torch.float32, "double*": torch.float64, "int*": torch.int32, "int32_t*": torch.int32,
             "int64_t*": torch.int64, "void*": None, "void**": None}


class Param(NamedTuple):
    name: str
    ctype: str            # normalised C type, e.g. "float*"
    pointer: bool
    dtype: torch.dtype | None     # dtype a tensor argument must have (None: any, or not a pointer)


class Prototype(NamedTuple):
    restype: type
    argtypes: tuple
    params: tuple         # of Param, the stream included


def _ctype(decl):
    return " ".join(re.sub(r"\bconst\b", " ", decl).split()).replace(" *", "*")


def parse_header(text):
    """{symbol: Prototype} of every gpz_* prototype in the text of a C header."""
    text = re.sub(r"/\*.*?\*/|//[^\n]*", " ", text, flags=re.S)
    text = re.sub(r"^\s*#.*$", " ", text, flags=re.M)
    protos = {}
    for stmt in re.split(r"[;{}]", text):
        stmt = " ".join(stmt.split())
        if "gpz_" not in stmt:
            continue
        m = re.fullmatch(r"(.+?)\b(gpz_\w+)\s*\((.*)\)", stmt)
        if m is None:
            raise GpzError(f"cannot read the prototype `{stmt}`")
        ret, sym, plist = m.groups()
        params = []
        for decl in ([] if plist.strip() in ("", "void") else plist.split(",")):
            pm = re.fullmatch(r"(.+[\s*])(\w+)", decl.strip())
            if pm is None:
                raise GpzError(f"cannot read the parameter `{decl.strip()}` of the prototype `{stmt}`")
            ct = _ctype(pm.group(1))
            if ct not in _SCALARS and ct not in _POINTERS:
                raise GpzError(f"unknown C type `{ct}` in the prototype `{stmt}`")
            params.append(Param(pm.group(2), ct, ct in _POINTERS, _POINTERS.get(ct)))
        ret = _ctype(ret)
        if ret not in _RESTYPES:
            raise GpzError(f"unknown C type `{ret}` in the prototype `{stmt}`")
        protos[sym] = Prototype(_RESTYPES[ret], tuple(ctypes.c_void_p if p.pointer else _SCALARS[p.ctype] for p in params),
                                tuple(params))
    return protos


_prototypes = None


def prototypes():
    """{symbol: Prototype} of include/gpzoo_b200.h (parsed once)."""
    global _prototypes
    if _prototypes is None:
        with open(HEADER) as f:
            _prototypes = parse_header(f.read())
    return _prototypes


class _Library(ctypes.CDLL):
    """The library whose symbols get the header's restype and argtypes at their first lookup (ctypes.CDLL keeps each looked-up
    function as an attribute).  A symbol the header does not declare stays untyped; a declared one that the library lacks
    raises AttributeError only when it is used."""

    def __getattr__(self, sym):
        fn = super().__getattr__(sym)
        proto = prototypes().get(sym)
        if proto is not None:
            fn.restype, fn.argtypes = proto.restype, proto.argtypes
        return fn


def lib():
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise GpzError(
                        f"{LIB_PATH} not found: build it with `python -m gpzoo_b200.build` "
                        "(gpzoo_b200 has no CPU or PyTorch fallback)")
                prototypes()                  # a header the binder cannot read fails here, at load
                _lib = _Library(LIB_PATH)
    return _lib


def _suffix(dtype):
    if dtype == torch.float32:
        return "f32"
    if dtype == torch.float64:
        return "f64"
    raise GpzError(f"gpzoo_b200 computes in float32 or float64, got {dtype}")


_launch_stream = None       # see launch_on()


def stream():
    if _launch_stream is not None:
        # side-stream launch: everything already queued on torch's current stream (the tensors' producers, and earlier users of
        # the recycled memory the outputs live in) is ordered before the kernel
        _launch_stream.wait_stream(torch.cuda.current_stream())
        return _launch_stream.cuda_stream
    return torch.cuda.current_stream().cuda_stream


class launch_on:
    """`with launch_on(side):` — C-ABI calls inside the block are launched on `side` while torch's current stream (and with it
    the caching allocator's stream of every tensor allocated inside) stays the same.  The caller joins with
    `torch.cuda.current_stream().wait_stream(side)` before anything consumes the outputs."""

    def __init__(self, st):
        self.st = st

    def __enter__(self):
        global _launch_stream
        self.prev, _launch_stream = _launch_stream, self.st

    def __exit__(self, *exc):
        global _launch_stream
        _launch_stream = self.prev


host_profile = None        # set to {} to record the longest host-side duration of every C-ABI call (debugging)
profile = None             # set to {} to record CUDA events around every C-ABI call (bench.py roofline numbers)


def kernel_launches():
    """Number of CUDA kernels the library has launched so far in this process."""
    return int(lib().gpz_launch_count())


_bound = {}                 # (name, dtype) -> (symbol, function, params)


def _bind(name, dtype):
    sym = f"gpz_{name}_{_suffix(dtype)}"
    proto = prototypes().get(sym)
    if proto is None:
        raise GpzError(f"{sym} is not declared in include/gpzoo_b200.h")
    b = _bound[(name, dtype)] = (sym, getattr(lib(), sym), proto.params)
    return b


def _device_pointer(sym, p, t):
    if not p.pointer:
        raise GpzError(f"{sym}: parameter {p.name} is {p.ctype}, got a tensor")
    if p.dtype is not None and t.dtype != p.dtype:
        raise GpzError(f"{sym}: parameter {p.name} is {p.ctype}, got a {t.dtype} tensor")
    if not t.is_cuda:
        raise GpzError("gpzoo_b200 kernels need CUDA tensors (no CPU path exists)")
    if not t.is_contiguous():
        raise GpzError("internal error: non-contiguous tensor passed to the C ABI")
    return t.data_ptr()


def call(name, dtype, *args):
    """Invoke gpz_<name>_<f32|f64>(*args, stream) and raise on a non-zero return code.

    `args` are checked against the header's prototype: one per parameter before the stream; a tensor goes to a pointer
    parameter of its dtype (void*: any dtype) and is passed as its device pointer; None is NULL; a ctypes array (a host table
    of pointers) passes as it is; ints and floats are converted to the parameter's C type by ctypes."""
    global launch_count
    sym, fn, params = _bound.get((name, dtype)) or _bind(name, dtype)
    if len(args) + 1 != len(params):
        raise GpzError(f"{sym} takes {len(params) - 1} arguments before the stream, got {len(args)}")
    args = list(args)
    for i, (a, p) in enumerate(zip(args, params)):
        if isinstance(a, torch.Tensor):
            args[i] = _device_pointer(sym, p, a)
        elif p.pointer and a is not None and not isinstance(a, ctypes.Array):
            raise GpzError(f"{sym}: parameter {p.name} is {p.ctype}, got {type(a).__name__} (a tensor or None is expected)")
    try:
        if profile is not None:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            st = stream()
            tst = _launch_stream if _launch_stream is not None else torch.cuda.current_stream()
            ev0.record(tst)
            rc = fn(*args, st)
            ev1.record(tst)
            profile.setdefault(name, []).append((ev0, ev1))
        elif host_profile is not None:          # debugging aid: host-side duration of every C-ABI call (longest call per name)
            import time
            t0 = time.perf_counter()
            rc = fn(*args, stream())
            dt_ms = (time.perf_counter() - t0) * 1e3
            host_profile[name] = max(host_profile.get(name, 0.0), dt_ms)
        else:
            rc = fn(*args, stream())
    except ctypes.ArgumentError as e:           # a value ctypes cannot convert to its parameter's C type
        p = params[int(re.match(r"argument (\d+)", str(e)).group(1)) - 1]
        raise GpzError(f"{sym}: parameter {p.name} ({p.ctype}): {e}") from None
    launch_count += 1
    if rc != 0:
        raise GpzError(f"{sym} failed: {lib().gpz_error_string(rc).decode()} (rc={rc})")


def exported_symbols():
    """Every symbol include/gpzoo_b200.h declares (used by the CPU test that the library exports them)."""
    return sorted(prototypes())
