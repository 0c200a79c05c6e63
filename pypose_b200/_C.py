"""ctypes binding of libb200pose.so — the C-ABI boundary (include/b200pose.h).

There is deliberately no CPU fallback: if the shared library is missing or a symbol cannot be
resolved, importing / calling raises.  PyTorch is used only for device memory and streams.
"""
import ctypes
import os

import torch

from ._optable import lie_symbols, lm_symbols, scan_symbols, knn_symbols, KNN_QUERIES

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libb200pose.so")

_lib = None
_fns = {}


class B200PoseError(RuntimeError):
    pass


def lib():
    """Load the shared library once (raises if it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B200PoseError(
                f"{LIB_PATH} not found: build it with `python -m pypose_b200._build` "
                "(pypose_b200 has no CPU/PyTorch fallback for its operators)")
        _lib = ctypes.CDLL(LIB_PATH)
    return _lib


def _bind(symbol, n_in, n_out, extra=()):
    f = getattr(lib(), symbol)
    f.restype = ctypes.c_int
    f.argtypes = [ctypes.c_void_p] * (n_in + n_out) + list(extra) + [ctypes.c_longlong, ctypes.c_void_p]
    return f


_LIE = {s: (ct, ins, outs) for s, ct, ins, outs, _ in lie_symbols()}
_LM = {s: args for s, args, _ in lm_symbols()}
_SCAN = {s: args for s, args, _ in scan_symbols()}
_KNN = {s: args for s, args, _ in knn_symbols()}
_QUERY = {s: (ret, args) for s, ret, args, _ in KNN_QUERIES}
_CT = {"double": ctypes.c_double, "int": ctypes.c_int, "long long": ctypes.c_longlong}


def fn(symbol):
    f = _fns.get(symbol)
    if f is None:
        if symbol in _LIE:
            _, ins, outs = _LIE[symbol]
            f = _bind(symbol, len(ins), len(outs))
        elif symbol in _LM:
            f = getattr(lib(), symbol)
            f.restype = ctypes.c_int
            f.argtypes = [ctypes.c_void_p if "*" in t else _CT[t] for t, _, _ in _LM[symbol]] + \
                [ctypes.c_longlong, ctypes.c_void_p]
        elif symbol in _SCAN or symbol in _KNN:
            f = getattr(lib(), symbol)
            f.restype = ctypes.c_int
            args = _SCAN[symbol] if symbol in _SCAN else _KNN[symbol]
            f.argtypes = [ctypes.c_void_p if "*" in t else _CT[t] for t, _, _ in args] + [ctypes.c_void_p]
        elif symbol in _QUERY:
            ret, args = _QUERY[symbol]
            f = getattr(lib(), symbol)
            f.restype = _CT[ret]
            f.argtypes = [ctypes.c_void_p if "*" in t else _CT[t] for t, _, _ in args]
        else:
            raise B200PoseError(f"unknown C-ABI symbol {symbol}")
        _fns[symbol] = f
    return f


def check(code, symbol):
    if code != 0:
        raise B200PoseError(f"{symbol} failed with CUDA error {code}")


_SFX = {torch.float32: "f32", torch.float64: "f64"}


def suffix(dtype):
    try:
        return _SFX[dtype]
    except KeyError:
        raise B200PoseError(f"b200pose kernels support float32/float64, got {dtype}") from None


def stream_ptr(device):
    return ctypes.c_void_p(torch._C._cuda_getCurrentRawStream(device.index if device.index is not None
                                                              else torch._C._cuda_getDevice()))


def enqueue(symbol, tensor, *args):
    """f(*args, stream) on `tensor`'s device and current stream.  The device guard is only entered when the current
    device differs (the context manager and `torch.cuda.current_stream` cost ~15 us per launch otherwise)."""
    f = _fns.get(symbol) or fn(symbol)
    idx = tensor.get_device()
    if idx == torch._C._cuda_getDevice():
        rc = f(*args, torch._C._cuda_getCurrentRawStream(idx))
    else:
        with torch.cuda.device(idx):
            rc = f(*args, torch._C._cuda_getCurrentRawStream(idx))
    if rc != 0:
        raise B200PoseError(f"{symbol} failed with CUDA error {rc}")


def launch_rows(base, ins, out_widths):
    """Run one elementwise Lie-op entry point `base`_{f32,f64} on (N, d) contiguous CUDA tensors."""
    x0 = ins[0]
    if not x0.is_cuda:
        raise B200PoseError(f"{base}: expected CUDA tensors (no CPU path), got device {x0.device}")
    for t in ins[1:]:       # every operand reaches the kernel as a raw pointer: same device and dtype or a clean error
        if t.device != x0.device or t.dtype != x0.dtype:
            raise B200PoseError(f"{base}: all operands must be on {x0.device} with dtype {x0.dtype}, got {t.device} / {t.dtype}")
    n = x0.shape[0]
    sym = f"{base}_{suffix(x0.dtype)}"
    outs = [torch.empty((n, w), dtype=x0.dtype, device=x0.device) for w in out_widths]
    if n == 0:
        return outs
    enqueue(sym, x0, *[t.data_ptr() for t in ins], *[t.data_ptr() for t in outs], n)
    return outs
