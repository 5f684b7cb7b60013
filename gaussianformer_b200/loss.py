"""Occupancy loss on the device: weighted cross-entropy + Lovász-softmax, forward and backward, with no host sync.

``OccupancyLoss`` keeps the reference's constructor kwargs and call signature (``loss/occupancy_loss.py:36-149``,
``loss/base_loss.py``) for the options the shipped configs use; ``occupancy_loss`` is the functional form.  The
arithmetic runs in the sm_100a kernels behind ``gf_occ_loss_forward`` (``include/gf_b200.h``): one C-ABI call computes
the loss and, when ``pred`` requires grad, the gradient, which the backward only scales by the upstream scalar.

Differences from the reference:

* equal Lovász errors are ordered by point index (a stable sort); the reference leaves their order to ``torch.sort``.
  The loss value does not depend on it, nor does the sum of the gradient over a group of tied errors of the same
  foreground status;
* the Lovász gradient of the Jaccard index is computed in closed form from integer counts (the reference subtracts
  fp32 Jaccard values near 1), and the loss is summed in fp64 in a fixed order: two calls give identical bits;
* a label that is neither a class nor ``ignore_index`` contributes nothing and, with ``validate``, raises
  ``ValueError`` (the reference hits a device-side assert);
* the parts ``loss_voxel_ce`` / ``loss_voxel_lovasz`` are returned detached, for logging; the gradient flows through
  the total.
"""
from __future__ import annotations

import ctypes
import os

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from ._lib import OccLossDesc
from .splat import _ptr, _require_cuda

IGNORE_INDEX = 255
_WS_BYTES = {}


def _workspace_bytes(desc):
    key = bytes(desc)
    n = _WS_BYTES.get(key)
    if n is None:
        L = _lib.lib()
        n = L.gf_occ_loss_workspace_bytes(ctypes.byref(desc))
        if n == 0:
            raise _lib.GfError(L.gf_last_error().decode())
        if len(_WS_BYTES) < 256:
            _WS_BYTES[key] = n
    return n


def occ_loss_raw(pred_nc, labels_u8, mask_u8, class_weights, *, use_softmax, ce_weight, lovasz_weight, lovasz_ignore,
                 ignore_empty, empty_label, lovasz=True, want_grad=True):
    """One ``gf_occ_loss_forward`` call on contiguous ``pred_nc [B,N,C]`` fp32, ``labels_u8 [B,N]``, ``mask_u8 [B,N]``
    (or None), ``class_weights [C]`` fp32 (or None).  Returns (loss3 [3], grad [B,N,C] or None, status [1] int32)."""
    B, N, C = pred_nc.shape
    dev = pred_nc.device
    d = OccLossDesc(B, N, C, int(bool(use_softmax)), IGNORE_INDEX, -1 if lovasz_ignore is None else int(lovasz_ignore),
                    int(bool(ignore_empty)), int(empty_label), float(ce_weight), float(lovasz_weight), int(bool(lovasz)))
    with torch.cuda.device(dev):
        ws_bytes = _workspace_bytes(d)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        loss3 = torch.empty(3, dtype=torch.float32, device=dev)
        status = torch.empty(1, dtype=torch.int32, device=dev)
        grad = torch.empty_like(pred_nc) if want_grad else None
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(_lib.lib().gf_occ_loss_forward(ctypes.byref(d), _ptr(pred_nc), _ptr(labels_u8), _ptr(mask_u8),
                                                  _ptr(class_weights), _ptr(loss3), _ptr(grad), _ptr(status),
                                                  _ptr(ws), ws_bytes, stream))
    return loss3, grad, status


class _OccLossFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, labels_u8, mask_u8, class_weights, opts):
        nc = pred.detach().transpose(1, 2)           # [B,N,C]: a view of the splat's logits, no copy
        if nc.dtype is not torch.float32 or not nc.is_contiguous():
            nc = nc.float().contiguous()
        loss3, grad, status = occ_loss_raw(nc, labels_u8, mask_u8, class_weights,
                                           want_grad=ctx.needs_input_grad[0], **opts)
        ctx.save_for_backward(grad)
        ctx.pred_dtype = pred.dtype
        ctx.mark_non_differentiable(status)
        return loss3, status

    @staticmethod
    def backward(ctx, g_loss3, _g_status):
        grad, = ctx.saved_tensors
        if grad is None:
            return None, None, None, None, None
        # only the total (entry 0) carries a gradient: the parts are handed out detached
        return (grad * g_loss3[0]).transpose(1, 2).to(ctx.pred_dtype), None, None, None, None


def occupancy_loss(pred, labels, occ_mask=None, class_weights=None, *, use_softmax=True, ce_weight=10.0,
                   lovasz_weight=1.0, lovasz_ignore=17, ignore_empty=False, empty_label=17, lovasz=True,
                   validate=None):
    """``OccupancyLoss.loss_voxel`` for one prediction (loss/occupancy_loss.py:102-149).

    ``pred [B,C,N]`` as ``GaussianHead`` hands it over (logits with ``use_softmax``, probabilities without);
    ``labels [B,N]`` any integer dtype, 255 = ignore; ``occ_mask [B,N]`` bool or None; ``class_weights [C]`` or None
    (ones).  All B samples form one pooled set.  Returns ``(loss, {"loss_voxel_ce": ..., "loss_voxel_lovasz": ...})``,
    device scalars.  ``validate`` (default: ``GF_B200_VALIDATE``, on unless "0") reads the status word back (one sync)
    and raises ``ValueError`` for labels that are neither a class nor 255."""
    _require_cuda(pred, labels, occ_mask)
    if pred.dim() != 3:
        raise ValueError(f"pred must be [B, C, N], got {tuple(pred.shape)}")
    B, C, N = pred.shape
    dev = pred.device
    lab = labels.reshape(B, N)
    lab = (lab if lab.dtype is torch.uint8 else lab.to(torch.uint8)).contiguous()
    mask = None
    if occ_mask is not None:
        mask = occ_mask.reshape(B, N)
        mask = (mask.view(torch.uint8) if mask.dtype is torch.bool else (mask != 0).view(torch.uint8)).contiguous()
    cw = None
    if class_weights is not None:
        cw = class_weights.to(device=dev, dtype=torch.float32).contiguous()
    opts = dict(use_softmax=use_softmax, ce_weight=ce_weight, lovasz_weight=lovasz_weight, lovasz_ignore=lovasz_ignore,
                ignore_empty=ignore_empty, empty_label=empty_label, lovasz=lovasz)
    loss3, status = _OccLossFunction.apply(pred, lab, mask, cw, opts)
    if validate is None:
        validate = os.environ.get("GF_B200_VALIDATE", "1") != "0"
    if validate and int(status.item()) & _lib.GF_OCC_LABEL_OUT_OF_RANGE:
        raise ValueError(f"labels outside 0..{C - 1} other than {IGNORE_INDEX}")
    return loss3[0], {"loss_voxel_ce": loss3[1].detach(), "loss_voxel_lovasz": loss3[2].detach()}


class OccupancyLoss(nn.Module):
    """Drop-in for the reference's registry-built ``OccupancyLoss`` (constructor kwargs of loss/occupancy_loss.py:36-100,
    ``forward(inputs)`` through ``input_dict`` as loss/base_loss.py).  The focal, dice and sem/geo-scal terms and the
    frequency-table class weights are not implemented (no shipped config enables them) and raise at construction."""

    def __init__(self, weight=1.0, empty_label=17, num_classes=18, use_focal_loss=False, focal_loss_args=None,
                 use_dice_loss=False, balance_cls_weight=False, multi_loss_weights=None, use_sem_geo_scal_loss=True,
                 use_lovasz_loss=True, lovasz_ignore=255, manual_class_weight=None, ignore_empty=False,
                 lovasz_use_softmax=True, input_dict=None, validate=None):
        super().__init__()
        if use_focal_loss:
            raise NotImplementedError("OccupancyLoss: use_focal_loss")
        if use_dice_loss:
            raise NotImplementedError("OccupancyLoss: use_dice_loss")
        if use_sem_geo_scal_loss:
            raise NotImplementedError("OccupancyLoss: use_sem_geo_scal_loss (pass use_sem_geo_scal_loss=False)")
        if balance_cls_weight and manual_class_weight is None:
            raise NotImplementedError("OccupancyLoss: balance_cls_weight without manual_class_weight")
        self.weight = weight
        self.input_dict = input_dict if input_dict is not None else {
            "pred_occ": "pred_occ", "sampled_xyz": "sampled_xyz", "sampled_label": "sampled_label",
            "occ_mask": "occ_mask"}
        self.empty_label = empty_label
        self.num_classes = num_classes
        self.use_lovasz_loss = use_lovasz_loss
        self.lovasz_ignore = lovasz_ignore
        self.ignore_empty = ignore_empty
        self.lovasz_use_softmax = lovasz_use_softmax
        mlw = multi_loss_weights or {}
        self.loss_voxel_ce_weight = mlw.get("loss_voxel_ce_weight", 1.0)
        self.loss_voxel_lovasz_weight = mlw.get("loss_voxel_lovasz_weight", 1.0)
        if balance_cls_weight:   # :82-88
            w = num_classes * F.normalize(torch.tensor(manual_class_weight, dtype=torch.float32), p=1, dim=-1)
        else:
            w = torch.ones(num_classes)
        self.register_buffer("class_weights", w)
        #: read the status word after each call and raise ValueError for out-of-range labels (one sync).
        self.validate = os.environ.get("GF_B200_VALIDATE", "1") != "0" if validate is None else validate
        _lib.lib()

    def forward(self, inputs):
        return self.weight * self.loss_voxel(**{k: inputs[v] for k, v in self.input_dict.items()})

    def loss_voxel(self, pred_occ, sampled_xyz, sampled_label, occ_mask=None):
        total = 0.
        for semantics in pred_occ:
            cw = self.class_weights
            if cw.device != semantics.device:
                cw = cw.to(semantics.device)
            loss, _ = occupancy_loss(semantics, sampled_label, occ_mask, cw, use_softmax=self.lovasz_use_softmax,
                                     ce_weight=self.loss_voxel_ce_weight, lovasz_weight=self.loss_voxel_lovasz_weight,
                                     lovasz_ignore=self.lovasz_ignore, ignore_empty=self.ignore_empty,
                                     empty_label=self.empty_label, lovasz=self.use_lovasz_loss,
                                     validate=self.validate)
            total = total + loss
        return total / len(pred_occ)
