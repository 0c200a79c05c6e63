"""k-nearest-neighbour search and the fused ICP correspondence step (csrc/knn.cu) as torch custom ops.

`ord` is passed as an integer code: 1, 2, or 0 for inf.  Batch dimensions broadcast; an operand whose batch has one
element reaches the kernel once with batch stride 0, so a cloud shared by every batch is never copied per batch.
"""
import ctypes
import math

import torch

from .. import _C
from ..lietensor.scan import _sms

NS = "b200pose"
torch.library.define(f"{NS}::knn", "(Tensor ref, Tensor nbr, int k, int ord, bool largest) -> (Tensor, Tensor)")
torch.library.define(f"{NS}::icp_moments", "(Tensor source, Tensor target, Tensor pose, int ord) -> Tensor")

NMOM = 17      # count, sum T s (3), sum t (3), sum t (T s)^T row-major (9), sum of distances


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _operand(x, batch):
    """(..., N, D) -> (contiguous tensor, batch stride in elements)."""
    N, D = x.shape[-2:]
    if math.prod(x.shape[:-2]) == 1:
        return x.reshape(N, D).contiguous(), 0
    if tuple(x.shape[:-2]) != tuple(batch):
        x = x.expand(*batch, N, D)
    return x.contiguous(), N * D


def _same_device(name, *ts):
    """Every operand reaches the kernel as a raw pointer: a tensor on another device must fail here, not in the kernel."""
    for t in ts[1:]:
        if t.device != ts[0].device:
            raise ValueError(f"{name}: all operands must be on {ts[0].device}, got {t.device}")


def _plan(B, N1, N2, k, x):
    splits = ctypes.c_longlong(0)
    nbytes = _C.fn("b200_knn_plan")(B, N1, N2, k, x.element_size(), _sms(x.device), ctypes.byref(splits))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device) if splits.value > 1 else None
    return splits.value, ws


@torch.library.impl(f"{NS}::knn", "CUDA")
def _knn_cuda(ref, nbr, k, ord, largest):
    _same_device("knn", ref, nbr)
    batch = torch.broadcast_shapes(ref.shape[:-2], nbr.shape[:-2])
    B, (N1, D), N2 = math.prod(batch), ref.shape[-2:], nbr.shape[-2]
    vals = torch.empty(*batch, N1, k, dtype=ref.dtype, device=ref.device)
    inds = torch.empty(*batch, N1, k, dtype=torch.int64, device=ref.device)
    if B * N1 == 0:
        return vals, inds
    r, rs = _operand(ref, batch)
    n, ns = _operand(nbr, batch)
    splits, ws = _plan(B, N1, N2, k, ref)
    sym = f"b200_knn_{_C.suffix(ref.dtype)}"
    with torch.cuda.device(ref.device):
        _C.check(_C.fn(sym)(_p(r), rs, _p(n), ns, B, N1, N2, D, k, ord, int(largest), splits, _p(ws), _p(vals), _p(inds),
                            _C.stream_ptr(ref.device)), sym)
    return vals, inds


@torch.library.register_fake(f"{NS}::knn")
def _knn_fake(ref, nbr, k, ord, largest):
    shape = (*torch.broadcast_shapes(ref.shape[:-2], nbr.shape[:-2]), ref.shape[-2], k)
    return ref.new_empty(shape), ref.new_empty(shape, dtype=torch.int64)


@torch.library.impl(f"{NS}::icp_moments", "CUDA")
def _icp_moments_cuda(source, target, pose, ord):
    """source (..., N1, 3), target (..., N2, 3), pose (batch, 7) in the source dtype -> (batch, NMOM) float64."""
    _same_device("icp_moments", source, target, pose)
    batch = pose.shape[:-1]
    B, N1, N2 = math.prod(batch), source.shape[-2], target.shape[-2]
    mom = torch.zeros(*batch, NMOM, dtype=torch.float64, device=source.device)
    if B * N1 == 0:
        return mom
    s, ss = _operand(source, batch)
    t, ts = _operand(target, batch)
    pose = pose.reshape(B, 7).contiguous()
    splits, ws = _plan(B, N1, N2, 1, source)
    sym = f"b200_icp_moments_{_C.suffix(source.dtype)}"
    with torch.cuda.device(source.device):
        _C.check(_C.fn(sym)(_p(s), ss, _p(t), ts, _p(pose), B, N1, N2, ord, splits, _p(ws), _p(mom),
                            _C.stream_ptr(source.device)), sym)
    return mom


@torch.library.register_fake(f"{NS}::icp_moments")
def _icp_moments_fake(source, target, pose, ord):
    return source.new_empty((*pose.shape[:-1], NMOM), dtype=torch.float64)
