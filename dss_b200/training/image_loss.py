"""The image objective of a DSS training step as one fused CUDA op (csrc/loss.cu, dss_dr_loss_forward / _backward).

``Trainer.calc_dr_loss`` (DSS/training/trainer.py:332-376) compares the rendered image with the data batch:

    L_rgb  = L1 over the rgb channels of the pixels where GT mask and rendered occupancy are both non-zero
             (channel sum, then the mean over those M pixels; 0 when M == 0)          L1Loss, losses.py:130-137
    L_mask = mean |mask - alpha|
    L_iou  = mean over views of 1 - sum(mask alpha) / eps_denom(sum(mask + alpha - mask alpha))    IouLoss, :498-514
    loss   = lambda_rgb L_rgb + lambda_silhouette (iou_weight L_iou + L_mask)

The reference selects the pixels with a boolean index and branches on ``mask_pred.sum() > 0`` in Python: two points per
step where the host waits for the device, and neither can be captured in a CUDA graph.  :func:`dr_image_loss` reads the
image and the batch's planes directly, reduces in a fixed order in fp64 and never reads anything back, so it is
bit-reproducible and capturable (dss_b200.graph.GraphedTrainStep captures it with the render step).
"""
import ctypes as C
from typing import NamedTuple

import torch

from .. import _lib

__all__ = ["DrLoss", "dr_image_loss"]


class DrLoss(NamedTuple):
    """0-d device tensors.  ``loss`` is differentiable with respect to the image; the three terms are detached and
    unweighted: ``loss_rgb`` is L_rgb and ``loss_silhouette`` is iou_weight L_iou + L_mask (multiply by lambda_rgb and
    lambda_silhouette for the reference's ``loss_dr_rgb`` and ``loss_dr_silhouette``)."""
    loss: torch.Tensor
    loss_rgb: torch.Tensor
    loss_silhouette: torch.Tensor
    loss_iou: torch.Tensor


def _args(image, img, mask, N, S, weights, partials, sums):
    a = _lib.DrLossArgs()
    a.image, a.img, a.mask = _lib.ptr(image), _lib.ptr(img), _lib.ptr(mask)
    a.n_views, a.image_size = N, S
    a.lambda_rgb, a.lambda_silhouette, a.iou_weight = weights
    a.partials, a.sums = _lib.ptr(partials), _lib.ptr(sums)
    return a


class _DrLossFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, image, img, mask, weights):
        dev = image.device
        image_c, img_c, mask_c = image.detach().contiguous(), img.detach().contiguous(), mask.detach().contiguous()
        N, S = image_c.shape[0], image_c.shape[1]
        f64 = dict(dtype=torch.float64, device=dev)
        partials = torch.empty((N * _lib.DR_LOSS_BLOCKS_PER_VIEW * _lib.DR_LOSS_NUM_SUMS,), **f64)
        sums = torch.empty((N + 1, _lib.DR_LOSS_NUM_SUMS), **f64)
        terms = torch.empty((4,), dtype=torch.float32, device=dev)
        a = _args(image_c, img_c, mask_c, N, S, weights, partials, sums)
        a.terms = _lib.ptr(terms)
        with torch.cuda.device(dev):
            rc = _lib.load().dss_dr_loss_forward(_lib.ctx(dev), C.byref(a), _lib.stream_ptr(dev))
        _lib.check(rc, "dss_dr_loss_forward")
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(image_c, img_c, mask_c, sums)
        ctx.weights = weights
        return terms

    @staticmethod
    def backward(ctx, grad_terms):
        if grad_terms is None:
            return None, None, None, None
        image_c, img_c, mask_c, sums = ctx.saved_tensors
        dev = image_c.device
        N, S = image_c.shape[0], image_c.shape[1]
        # only terms[0] (the loss) reaches the caller undetached, so grad_terms[0] is the whole upstream gradient
        grad_terms = _lib.as_f32(grad_terms, "grad_loss")
        grad_image = torch.empty_like(image_c)
        a = _args(image_c, img_c, mask_c, N, S, ctx.weights, None, sums)
        a.grad_loss, a.grad_image = _lib.ptr(grad_terms), _lib.ptr(grad_image)
        with torch.cuda.device(dev):
            rc = _lib.load().dss_dr_loss_backward(_lib.ctx(dev), C.byref(a), _lib.stream_ptr(dev))
        _lib.check(rc, "dss_dr_loss_backward")
        return grad_image, None, None, None


def _dr_terms(image, img, mask, lambda_rgb, lambda_silhouette, iou_weight):
    """checked call of the op: the (4,) terms {loss, rgb, silhouette, iou}, differentiable through element 0 only"""
    _lib.require_cuda(image, img, mask)
    for name, t in (("image", image), ("img", img), ("mask", mask)):
        _lib.as_f32(t, name)
    if image.dim() != 4 or image.shape[3] != 4 or image.shape[1] != image.shape[2]:
        raise RuntimeError("image must have shape (N,S,S,4), got %s" % (tuple(image.shape),))
    N, S = int(image.shape[0]), int(image.shape[1])
    if N < 1 or S < 1:
        raise RuntimeError("image must hold at least one pixel, got %s" % (tuple(image.shape),))
    if tuple(img.shape) != (N, 3, S, S):
        raise RuntimeError("img must have shape (%d, 3, %d, %d), got %s" % (N, S, S, tuple(img.shape)))
    if tuple(mask.shape) not in ((N, 1, S, S), (N, S, S)):
        raise RuntimeError("mask must have shape (%d, 1, %d, %d) or (%d, %d, %d), got %s"
                           % (N, S, S, N, S, S, tuple(mask.shape)))
    weights = (float(lambda_rgb), float(lambda_silhouette), float(iou_weight))
    if min(weights[:2]) < 0:
        raise ValueError("lambda_rgb and lambda_silhouette must be >= 0")
    return _DrLossFunction.apply(image, img, mask, weights)


def dr_image_loss(image, img, mask, lambda_rgb=1.0, lambda_silhouette=1.0, iou_weight=0.01) -> DrLoss:
    """Image objective of ``Trainer.calc_dr_loss`` on the device, without a host wait.

    image : (N,S,S,4) float32 rendered rgb + occupancy (``render_points(...).image``)
    img   : (N,3,S,S) float32 ground-truth colours, as the data batch holds them
    mask  : (N,1,S,S) or (N,S,S) float32 ground-truth mask (values need not be binary)
    The lambdas are the trainer's ``lambda_dr_rgb`` / ``lambda_dr_silhouette``; a term whose lambda is 0 contributes
    neither value nor gradient to ``loss``, as in the reference (which skips it).
    """
    terms = _dr_terms(image, img, mask, lambda_rgb, lambda_silhouette, iou_weight)
    parts = terms.detach()
    return DrLoss(terms[0], parts[1], parts[2], parts[3])
