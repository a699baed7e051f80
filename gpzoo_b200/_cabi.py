"""ctypes binding of include/gpzoo_b200.h.

The CUDA shared library is the product: if it is missing or a call fails, this module raises — there is
no PyTorch / CPU fallback anywhere in the package.
"""
from __future__ import annotations

import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GPZ_LIB") or os.path.join(_HERE, "lib", "libgpzoo_b200.so")     # GPZ_LIB: A/B runs of two builds
_lib = None
_lock = threading.Lock()
launch_count = 0          # number of C-ABI compute calls issued (bench.py reports kernel launches from this)

c_i, c_i64, c_f, c_d, c_p = ctypes.c_int, ctypes.c_int64, ctypes.c_float, ctypes.c_double, ctypes.c_void_p


class GpzError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise GpzError(
                        f"{LIB_PATH} not found: build it with `python -m gpzoo_b200.build` "
                        "(gpzoo_b200 has no CPU or PyTorch fallback)")
                l = ctypes.CDLL(LIB_PATH)
                l.gpz_error_string.restype = ctypes.c_char_p
                l.gpz_error_string.argtypes = [c_i]
                l.gpz_abi_version.restype = c_i
                l.gpz_launch_count.restype = ctypes.c_longlong
                for suf in ("f32", "f64"):
                    getattr(l, f"gpz_poisson_workspace_bytes_{suf}").restype = c_i64
                    getattr(l, f"gpz_poisson_csc_workspace_bytes_{suf}").restype = c_i64
                    getattr(l, f"gpz_negbin_workspace_bytes_{suf}").restype = c_i64
                _lib = l
    return _lib


def _suffix(dtype):
    if dtype == torch.float32:
        return "f32", c_f
    if dtype == torch.float64:
        return "f64", c_d
    raise GpzError(f"gpzoo_b200 computes in float32 or float64, got {dtype}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL).  Tensors must be contiguous CUDA tensors."""
    if t is None:
        return c_p(0)
    if not t.is_cuda:
        raise GpzError("gpzoo_b200 kernels need CUDA tensors (no CPU path exists)")
    if not t.is_contiguous():
        raise GpzError("internal error: non-contiguous tensor passed to the C ABI")
    return c_p(t.data_ptr())


_launch_stream = None       # see launch_on()


def stream():
    if _launch_stream is not None:
        # side-stream launch: everything already queued on torch's current stream (the tensors' producers, and earlier users of
        # the recycled memory the outputs live in) is ordered before the kernel
        _launch_stream.wait_stream(torch.cuda.current_stream())
        return c_p(_launch_stream.cuda_stream)
    return c_p(torch.cuda.current_stream().cuda_stream)


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


def call(name, dtype, *args):
    """Invoke gpz_<name>_<f32|f64>(*args, stream) and raise on a non-zero return code."""
    global launch_count
    suf, _ = _suffix(dtype)
    fn = getattr(lib(), f"gpz_{name}_{suf}")
    if fn.restype is not c_i:
        fn.restype = c_i
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
    launch_count += 1
    if rc != 0:
        raise GpzError(f"gpz_{name}_{suf} failed: {lib().gpz_error_string(rc).decode()} (rc={rc})")


def scalar(dtype, v):
    return _suffix(dtype)[1](float(v))


def exported_symbols():
    """Every symbol include/gpzoo_b200.h declares (used by the CPU test that the library exports them)."""
    import re
    hdr = os.path.join(os.path.dirname(_HERE), "include", "gpzoo_b200.h")
    txt = open(hdr).read()
    return sorted(set(re.findall(r"\b(gpz_[a-z0-9_]+)\s*\(", txt)))
