"""B200-native drop-in for the reference's model/chamfer.py (SURVEY.md section 8, row f-4).

chamfer_batch(p1 [B,N,D], p2 [B,M,D]) = sum over b, n of min_m ||p1[b,n] - p2[b,m]||_2, divided by B (chamfer.py:32-53);
chamfer_non_batch is the same for B == 1 without the division (:7-30).  One kernel (pn_chamfer_f32): no [B,N,M,D] cube.
The reference's only known-answer check lives in this file (`__main__`, :55-67: 11.6073 twice); tests/ repeats it.

Differentiable like the reference's norm -> min -> sum: with grad mode on and a cloud that requires a gradient, the forward
also keeps each p1 point's nearest p2 point (pn_chamfer_argmin_f32) and the result carries a grad_fn whose backward is
pn_chamfer_bwd_f32 (pointnet12_b200/train.ChamferFn).  Otherwise the forward-only kernel runs and nothing is kept.
"""
import torch

from .. import _native as nv
from .. import ops
from .pointnet_util import grad_path


def _chamfer_sum(p1: torch.Tensor, p2: torch.Tensor) -> torch.Tensor:
    p1, p2 = ops._cloud(p1, "p1"), ops._cloud(p2, "p2")
    assert p1.size(0) == p2.size(0) and p1.size(2) == p2.size(2)
    B, N, D = p1.shape
    total = torch.empty((1,), dtype=torch.float64, device=p1.device)
    with ops._on_device(p1):
        nv.call("pn_chamfer_f32", p1.data_ptr(), *p1.stride(), p2.data_ptr(), *p2.stride(), B, N, p2.shape[1], D, None,
                total.data_ptr(), ops._stream())
    return total[0]


def chamfer_non_batch(p1: torch.Tensor, p2: torch.Tensor) -> torch.Tensor:
    assert p1.size(0) == 1 and p2.size(0) == 1
    if grad_path(p1, p2):
        from ..train import ChamferFn
        return ChamferFn.apply(p1, p2, 1)
    return _chamfer_sum(p1, p2).to(torch.float32)


def chamfer_batch(p1: torch.Tensor, p2: torch.Tensor) -> torch.Tensor:
    if grad_path(p1, p2):
        from ..train import ChamferFn
        return ChamferFn.apply(p1, p2, p1.size(0))
    return (_chamfer_sum(p1, p2) / p1.size(0)).to(torch.float32)
