"""Projection / reprojection residual models (reference: pypose/function/geometry.py:7-225).

Only the camera-model functions the LM configs use are in scope (SURVEY.md §2 row 12), plus `svdtf`, which EPnP
(SURVEY.md §8f.4, module/pnp.py) and ICP need, and `knn` (csrc/knn.cu); the point-cloud filters are not built.
"""
import math

import torch

from ..basics import pm
from .checking import is_lietensor
from . import _knn  # noqa: F401  (defines b200pose::knn and b200pose::icp_moments)


def cart2homo(coordinates: torch.Tensor):
    """Append a homogeneous 1 (geometry.py:7-34)."""
    return torch.cat([coordinates, torch.ones_like(coordinates[..., :1])], dim=-1)


def homo2cart(coordinates: torch.Tensor):
    """Divide by the last coordinate, sign-preserving clamp away from 0 (geometry.py:37-57)."""
    last = coordinates[..., -1:]
    denom = pm(last) * last.abs().clamp_(min=torch.finfo(coordinates.dtype).tiny)
    return coordinates[..., :-1] / denom


def point2pixel(points, intrinsics, extrinsics=None):
    """Pinhole projection of (..., N, 3) points with (..., 3, 3) intrinsics (geometry.py:60-112)."""
    assert points.size(-1) == 3, "Points shape incorrect"
    assert intrinsics.size(-1) == intrinsics.size(-2) == 3, "Intrinsics shape incorrect."
    if extrinsics is None:
        torch.broadcast_shapes(points.shape[:-2], intrinsics.shape[:-2])
    else:
        assert is_lietensor(extrinsics) and extrinsics.shape[-1] == 7, "Type incorrect."
        torch.broadcast_shapes(points.shape[:-2], intrinsics.shape[:-2], extrinsics.shape[:-1])
        points = extrinsics.unsqueeze(-2) @ points
    return homo2cart(points @ intrinsics.mT)


def pixel2point(pixels, depth, intrinsics):
    """Back-projection of (..., N, 2) pixels with (..., N) depths through (..., 3, 3) pinhole intrinsics to (..., N, 3)
    camera-frame points: z = depth, x = (u - cx) z / fx, y = (v - cy) z / fy (geometry.py:115-168)."""
    assert pixels.size(-1) == 2, "Pixels shape incorrect"
    assert depth.size(-1) == pixels.size(-2), "Depth shape does not match pixels"
    assert intrinsics.size(-1) == intrinsics.size(-2) == 3, "Intrinsics shape incorrect."
    focal = torch.stack([intrinsics[..., 0, 0], intrinsics[..., 1, 1]], dim=-1)
    assert not torch.any(focal == 0), "fx / fy cannot contain zero"
    centre = intrinsics[..., :2, 2]
    xy = (pixels - centre.unsqueeze(-2)) * depth.unsqueeze(-1) / focal.unsqueeze(-2)
    return torch.cat([xy, depth.unsqueeze(-1)], dim=-1)


def reprojerr(points, pixels, intrinsics, extrinsics=None, reduction='none'):
    """Per-pixel reprojection error (geometry.py:171-225)."""
    torch.broadcast_shapes(points.shape[:-2], pixels.shape[:-2], intrinsics.shape[:-2])
    assert points.size(-1) == 3 and pixels.size(-1) == 2 and \
        intrinsics.size(-1) == intrinsics.size(-2) == 3, "Shape not compatible."
    assert reduction in {'norm', 'sum', 'none'}, "Reduction method can only be 'norm'|'sum'|'none'."
    err = point2pixel(points, intrinsics, extrinsics) - pixels
    if reduction == 'norm':
        return err.norm(dim=-1)
    if reduction == 'sum':
        return err.sum(dim=-1)
    return err


def svdtf(source, target):
    """Rigid alignment of two associated point sets (..., N, 3) -> SE3 `T` with `T @ source ~ target`
    (geometry.py:315-358): rotation from the SVD of the cross-covariance of the centred sets.  Kept quirk: an improper
    solution (det = -1) is negated as a whole, as the reference does (:353-354), not by flipping one singular vector."""
    assert source.size(-2) == target.size(-2), "The number of points N has to be the same for both point clouds."
    cs, ct = source.mean(dim=-2, keepdim=True), target.mean(dim=-2, keepdim=True)
    cov = (target - ct).mT @ (source - cs)                       # (..., 3, 3): sum_n target_n source_n^T
    return rigid_from_moments(cs, ct, cov)


def rigid_from_moments(cs, ct, cov):
    """The SE3 of `svdtf` from the centroids `cs`, `ct` (..., 1, 3) of the source and target sets and their centred
    cross-covariance `cov` (..., 3, 3) = sum_n (t_n - ct)(s_n - cs)^T.  ICP forms these from fp64 moments."""
    from ..lietensor import mat2SE3
    U, _, Vh = torch.linalg.svd(cov)
    R = U @ Vh
    improper = (torch.linalg.det(R) + 1).abs() < 1e-6
    R = torch.where(improper[..., None, None], -R, R)
    t = ct.mT - R @ cs.mT
    return mat2SE3(torch.cat([R, t], dim=-1), check=False)


_ORD = {1: 1, 2: 2, math.inf: 0}
KNN_MAX_D, KNN_MAX_K = 8, 32


def knn_ord_code(ord):
    """The kernels' code for the norm order: 1, 2, or 0 for inf; anything else raises ValueError."""
    try:
        return _ORD[ord]
    except (KeyError, TypeError):
        raise ValueError(f"knn: ord must be 1, 2 or inf, got {ord!r}") from None


def knn(ref, nbr, k=1, ord=2, dim=-1, largest=False, sorted=True):
    r"""The k nearest (or, with ``largest``, furthest) points of ``nbr`` to each point of ``ref``
    (reference: pypose/function/geometry.py:228-313).

    Args:
        ref (``torch.Tensor``): reference points, shape (..., N1, D).
        nbr (``torch.Tensor``): neighbour points, shape (..., N2, D); the batch dimensions broadcast with ``ref``'s.
        k (``int``): number of neighbours, 1 <= k <= min(32, N2). Default: 1.
        ord (``int``): norm of the difference: 1, 2 or ``inf``. Default: 2.
        dim (``int``): the coordinate dimension; only the last one (-1, or ``ref.dim() - 1``) is supported.
        largest (``bool``): return the furthest points instead of the nearest. Default: ``False``.
        sorted (``bool``): accepted for compatibility; results are always sorted.

    Returns:
        ``torch.return_types.topk(values (..., N1, k), indices (..., N1, k) int64)``: ``values`` are the ``ord``-norm
        distances (not squared), differentiable with respect to ``ref`` and ``nbr``; ``indices`` index ``nbr``.

    The search runs on the GPU (csrc/knn.cu) for float32 and float64 CUDA tensors with 1 <= D <= 8; other inputs
    raise ``ValueError``, as do ``ref`` and ``nbr`` on different devices; CPU tensors raise, as every other op of
    the package does.  Unlike the reference, memory is
    O(N1 k), not O(N1 N2 D).  Results are sorted ascending (descending with ``largest``) whatever ``sorted`` says,
    equal distances are ordered by the lower ``nbr`` index, and a NaN distance orders above every finite one.
    """
    if not (torch.is_tensor(ref) and torch.is_tensor(nbr)):
        raise ValueError("knn: ref and nbr must be tensors")
    if ref.dtype not in (torch.float32, torch.float64) or nbr.dtype != ref.dtype:
        raise ValueError(f"knn: ref and nbr must both be float32 or both float64, got {ref.dtype} / {nbr.dtype}")
    if ref.device != nbr.device:
        raise ValueError(f"knn: ref and nbr must be on the same device, got {ref.device} / {nbr.device}")
    if ref.dim() < 2 or nbr.dim() < 2:
        raise ValueError("knn: ref and nbr must have shape (..., N, D)")
    if dim not in (-1, ref.dim() - 1):
        raise ValueError(f"knn: only the last dimension can hold the coordinates (dim=-1), got dim={dim}")
    D = ref.shape[-1]
    if nbr.shape[-1] != D:
        raise ValueError(f"knn: ref and nbr must have the same point dimension, got {D} and {nbr.shape[-1]}")
    if not 1 <= D <= KNN_MAX_D:
        raise ValueError(f"knn: the point dimension D must be in 1..{KNN_MAX_D}, got {D}")
    N2 = nbr.shape[-2]
    if not isinstance(k, int) or not 1 <= k <= min(KNN_MAX_K, N2):
        raise ValueError(f"knn: k must be in 1..min({KNN_MAX_K}, N2={N2}), got {k}")
    if N2 >= 2 ** 31:
        raise ValueError(f"knn: N2 must be below 2^31, got {N2}")
    code = knn_ord_code(ord)
    try:
        torch.broadcast_shapes(ref.shape[:-2], nbr.shape[:-2])
    except RuntimeError as e:
        raise ValueError(f"knn: batch dimensions do not broadcast: {e}") from None
    values, indices = _KNN.apply(ref, nbr, k, code, bool(largest))
    return torch.return_types.topk((values, indices))


class _KNN(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ref, nbr, k, code, largest):
        values, indices = torch.ops.b200pose.knn(ref, nbr, k, code, largest)
        ctx.save_for_backward(ref, nbr, values, indices)
        ctx.code = code
        ctx.mark_non_differentiable(indices)
        return values, indices

    @staticmethod
    def backward(ctx, gv, _):
        """O(N1 k): the neighbours are gathered from the saved indices; at zero distance the gradient is 0, as for
        torch.linalg.vector_norm."""
        ref, nbr, values, indices = ctx.saved_tensors
        batch, (N1, k), (N2, D) = values.shape[:-2], values.shape[-2:], nbr.shape[-2:]
        flat = indices.reshape(*batch, N1 * k, 1).expand(*batch, N1 * k, D)
        diff = ref.unsqueeze(-2) - torch.gather(nbr.expand(*batch, N2, D), -2, flat).reshape(*batch, N1, k, D)
        v = values.unsqueeze(-1)
        if ctx.code == 2:
            w = torch.where(v == 0, torch.zeros_like(diff), diff / v)
        elif ctx.code == 1:
            w = diff.sign()
        else:                                   # inf: shared between the coordinates that attain the max
            hit = (diff.abs() == v).to(diff.dtype)
            w = diff.sign() * hit / hit.sum(-1, keepdim=True).clamp(min=1)
        gw = gv.unsqueeze(-1) * w               # (..., N1, k, D) gradient with respect to the difference
        gref = gnbr = None
        if ctx.needs_input_grad[0]:
            gref = gw.sum(-2).sum_to_size(ref.shape)
        if ctx.needs_input_grad[1]:
            B = math.prod(batch)
            offs = (torch.arange(B, device=indices.device) * N2).view(*batch, 1, 1) if batch else 0
            g = torch.zeros(B * N2, D, dtype=gw.dtype, device=gw.device)
            g.index_add_(0, (indices + offs).reshape(-1), gw.reshape(-1, D), alpha=-1)
            gnbr = g.view(*batch, N2, D).sum_to_size(nbr.shape)
        return gref, gnbr, None, None, None
