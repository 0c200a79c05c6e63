"""Batched iterative closest point (reference: pypose/module/icp.py).

Each iteration is one fused kernel (b200pose::icp_moments, csrc/knn.cu): the source cloud is transformed by the current
estimate on the fly, each point is matched to its nearest target point and the per-batch fp64 moments of the matches
are accumulated.  The 3x3 alignment of those moments is the one `svdtf` computes (`rigid_from_moments`), and the
estimate is composed as T <- dT T instead of re-transforming the cloud.
"""
import torch
from torch import nn

from ..function.checking import is_lietensor, is_SE3
from ..function.geometry import knn_ord_code, rigid_from_moments
from ..utils.stepper import ReduceToBason


class ICP(nn.Module):
    r'''Batched ICP: the SE3 transform :math:`T` that minimises :math:`\sum_i \|p_{\mathrm{target},j(i)} - T
    p_{\mathrm{source},i}\|`, where :math:`j(i)` is the nearest target point of the transformed source point.

    Args:
        init (``LieTensor``, optional): initial SE3 transform. Default: ``None`` (identity).
        stepper (optional): decides when to stop; ``pypose_b200.utils.ReduceToBason(steps=200)`` if ``None``.

    The error handed to the stepper at each iteration is the mean nearest-neighbour distance of each batch, measured
    before that iteration's update.
    '''
    def __init__(self, init=None, stepper=None):
        super().__init__()
        _check_se3(init)
        self.init = init
        self.stepper = stepper if stepper is not None else ReduceToBason(steps=200)

    def forward(self, source, target, ord=2, dim=-1, init=None):
        r'''
        Args:
            source (``torch.Tensor``): source clouds (..., N1, 3).
            target (``torch.Tensor``): target clouds (..., N2, 3); the batch dimensions broadcast with the source's.
            ord (``int``, optional): norm used for the nearest-neighbour distance: 1, 2 or ``inf``. Default: 2.
            dim (``int``, optional): the coordinate dimension; only -1 is supported. Default: -1.
            init (``LieTensor``, optional): initial SE3 transform, overriding the constructor's. Default: ``None``.

        Returns:
            ``LieTensor``: the SE3 transform from source to target, with the broadcast batch shape.
        '''
        from ..lietensor import SE3
        code = knn_ord_code(ord)
        if dim not in (-1, source.dim() - 1):
            raise ValueError(f"ICP: only the last dimension can hold the coordinates (dim=-1), got dim={dim}")
        if source.dim() < 2 or target.dim() < 2 or source.size(-1) != 3 or target.size(-1) != 3:
            raise ValueError("ICP: source and target must have shape (..., N, 3)")
        if source.size(-2) == 0 or target.size(-2) == 0:
            raise ValueError("ICP: source and target must hold at least one point each")
        if source.dtype not in (torch.float32, torch.float64) or target.dtype != source.dtype:
            raise ValueError(f"ICP: source and target must both be float32 or both float64, got "
                             f"{source.dtype} / {target.dtype}")
        if source.device != target.device:
            raise ValueError(f"ICP: source and target must be on the same device, got {source.device} / {target.device}")
        start = self.init if init is None else init
        _check_se3(start)
        shapes = [source.shape[:-2], target.shape[:-2]] + ([] if start is None else [start.shape[:-1]])
        try:
            batch = torch.broadcast_shapes(*shapes)
        except RuntimeError as e:
            raise ValueError(f"ICP: batch dimensions do not broadcast: {e}") from None
        identity = torch.tensor([0.0] * 6 + [1.0], dtype=torch.float64, device=source.device)
        T = identity if start is None else start.tensor().to(device=source.device, dtype=torch.float64)
        T = SE3(T.expand(*batch, 7).contiguous())
        self.stepper.reset()
        while self.stepper.continual():
            mom = torch.ops.b200pose.icp_moments(source, target, T.tensor().to(source.dtype), code)
            n = mom[..., :1]
            cs, ct = mom[..., 1:4] / n, mom[..., 4:7] / n
            cov = mom[..., 7:16].unflatten(-1, (3, 3)) - n.unsqueeze(-1) * ct.unsqueeze(-1) * cs.unsqueeze(-2)
            error = (mom[..., 16] / n[..., 0]).to(source.dtype)
            T = rigid_from_moments(cs.unsqueeze(-2), ct.unsqueeze(-2), cov) @ T
            self.stepper.step(error)
        return SE3(T.tensor().to(source.dtype))


def _check_se3(init):
    if init is not None and not (is_lietensor(init) and is_SE3(init)):
        raise ValueError(f"ICP: the initial transform must be an SE3 LieTensor, got {type(init).__name__}")
