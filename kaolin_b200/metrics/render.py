"""``mask_iou`` — drop-in for kaolin/metrics/render.py:18-41, the silhouette loss the DIB-R loop
applies to the soft mask (SURVEY.md §8f rank 2): the per-view sums of ``lhs*rhs`` and
``lhs+rhs-lhs*rhs`` in one streaming pass and an element-wise backward
(kaolin_b200/csrc/mesh_pipeline.cu) instead of ~8 PyTorch kernels with full-image temporaries."""
import torch
from torch.autograd import Function

from .. import _lib
from ..render.mesh import _host

__all__ = ["mask_iou"]


class MaskIouB200(Function):
    @staticmethod
    def forward(ctx, lhs_mask, rhs_mask):
        l, r = _host.aligned(lhs_mask.contiguous()), _host.aligned(rhs_mask.contiguous())
        B = l.shape[0]
        hw = l.numel() // B
        sums = torch.empty((B, 2), dtype=torch.float32, device=l.device)
        loss = torch.empty((), dtype=torch.float32, device=l.device)
        with torch.cuda.device(l.device):
            st = _lib.lib().dibr_b200_mask_iou_forward(B, hw, _host.ptr(l), _host.ptr(r), _host.ptr(sums),
                                                       _host.ptr(loss), _host.stream_ptr(l.device))
        _lib.check(st, "dibr_b200_mask_iou_forward")
        ctx.save_for_backward(l, r, sums)
        return loss

    @staticmethod
    def backward(ctx, g_loss):
        l, r, sums = ctx.saved_tensors
        B = l.shape[0]
        hw = l.numel() // B
        g_l = torch.empty_like(l) if ctx.needs_input_grad[0] else None
        g_r = torch.empty_like(r) if ctx.needs_input_grad[1] else None
        g = _host.aligned(g_loss.contiguous().to(torch.float32))
        with torch.cuda.device(l.device):
            st = _lib.lib().dibr_b200_mask_iou_backward(B, hw, _host.ptr(l), _host.ptr(r), _host.ptr(sums),
                                                        _host.ptr(g), _host.ptr(g_l), _host.ptr(g_r),
                                                        _host.stream_ptr(l.device))
        _lib.check(st, "dibr_b200_mask_iou_backward")
        return g_l, g_r


def mask_iou(lhs_mask, rhs_mask):
    r"""IoU loss of two segmentation masks of shape (batch_size, height, width):
    ``1 - mean_b( sum(l*r) / (sum(l + r - l*r) + 1e-10) )`` (kaolin.metrics.render.mask_iou)."""
    _host.check_tensors("mask_iou", [("lhs_mask", lhs_mask), ("rhs_mask", rhs_mask)])
    if lhs_mask.dim() != 3:
        raise RuntimeError("mask_iou: masks must be of shape (batch_size, height, width)")
    assert rhs_mask.shape == lhs_mask.shape
    return MaskIouB200.apply(lhs_mask, rhs_mask)
