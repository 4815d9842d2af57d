"""Drop-in for the ``nn.CrossEntropyLoss()`` the reference builds at main.py:99 and calls at
train.py:37: same constructor arguments and ``__call__(outputs, targets)``; forward and
d(loss)/d(logits) come from ONE fused kernel (csrc/softmax_ce.cu, csrc/softmax_ce_ex.cu)."""
from __future__ import annotations

import warnings
from typing import Optional

import torch
import torch.nn as nn

from . import ops

_REDUCTIONS = ("mean", "sum", "none")


class _FusedCE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, target):
        need = logits.requires_grad
        loss, dl = ops.softmax_ce(logits.contiguous(), target.contiguous(), want_grad=need)
        ctx.dl = dl
        return loss

    @staticmethod
    def backward(ctx, gout):
        dl, ctx.dl = ctx.dl, None
        if (gout.is_cuda and gout.numel() == 1 and gout.dtype == torch.float32 and dl.numel() % 4 == 0
                and not torch.is_grad_enabled()):
            # loss.backward(): gout is ones -- scale in place on the device only if it is not (no 2 x 168 MB elementwise pass)
            ops.scale_unless_one(dl, gout)
            return dl, None
        return dl * gout, None


class _FusedCEEx(torch.autograd.Function):
    """The loss with its options.  'mean' / 'sum': forward and gradient in one pass, as _FusedCE.  'none': the forward
    writes the loss map; the backward re-reads logits and targets and writes d(logits) for the incoming per-pixel gradient
    in one pass."""

    @staticmethod
    def forward(ctx, logits, target, weight, ignore_index, label_smoothing, reduction):
        logits, target = logits.contiguous(), target.contiguous()
        if reduction == "none":
            loss, _ = ops.softmax_ce_ex(logits, target, weight, ignore_index, label_smoothing, "none")
            ctx.save_for_backward(logits, target, weight)
            ctx.opts = (ignore_index, label_smoothing)
            ctx.dl = None
            return loss
        loss, dl = ops.softmax_ce_ex(logits, target, weight, ignore_index, label_smoothing, reduction,
                                     want_grad=logits.requires_grad)
        ctx.dl = dl
        return loss

    @staticmethod
    def backward(ctx, gout):
        if ctx.dl is None:
            logits, target, weight = ctx.saved_tensors
            ignore_index, label_smoothing = ctx.opts
            dl = ops.softmax_ce_ex_backward(logits, target, gout.float().contiguous(), weight, ignore_index, label_smoothing)
            return dl, None, None, None, None, None
        dl, ctx.dl = ctx.dl, None
        if (gout.is_cuda and gout.numel() == 1 and gout.dtype == torch.float32 and dl.numel() % 4 == 0
                and not torch.is_grad_enabled()):
            ops.scale_unless_one(dl, gout)
            return dl, None, None, None, None, None
        return dl * gout, None, None, None, None, None


class CrossEntropyLoss(nn.Module):
    """``torch.nn.CrossEntropyLoss`` over NCHW f32 logits ``[B,C,H,W]`` (other float dtypes are converted) and class-index
    targets ``[B,H,W]`` of int64 or uint8, on CUDA.

    The arguments mean what they mean in torch: ``weight`` (C per-class weights, registered as the buffer ``weight`` so
    that ``.to()`` moves it and ``state_dict()`` holds it), ``ignore_index``, ``reduction`` ('mean' divides by the weight
    sum of the counted targets; 'none' returns the ``[B,H,W]`` loss map) and ``label_smoothing`` in [0, 1].  A uint8 label
    equals ``ignore_index`` only when ``ignore_index`` is in [0, 255].  The deprecated ``size_average`` / ``reduce`` are
    mapped to ``reduction`` as torch maps them, with torch's warning.  Class-probability targets are not supported.

    Unlike torch, a label outside [0, C) that is not ``ignore_index`` does not raise (that would need a host sync): the loss
    is NaN ('none': at those pixels) and those pixels get no gradient.

    With every argument at its default and int64 targets the call runs the original fused kernel (csrc/softmax_ce.cu);
    anything else runs csrc/softmax_ce_ex.cu.  Neither synchronises with the host, so both can be captured in a CUDA graph.
    """

    def __init__(self, weight: Optional[torch.Tensor] = None, size_average=None, ignore_index: int = -100, reduce=None,
                 reduction: str = "mean", label_smoothing: float = 0.0) -> None:
        super().__init__()
        if size_average is not None or reduce is not None:
            reduction = _legacy_reduction(size_average, reduce)
        if reduction not in _REDUCTIONS:
            raise ValueError(f"{reduction} is not a valid value for reduction")
        label_smoothing = float(label_smoothing)
        if not 0.0 <= label_smoothing <= 1.0:
            raise RuntimeError(f"label_smoothing must be between 0.0 and 1.0. Got: {label_smoothing}")
        if weight is not None and (not isinstance(weight, torch.Tensor) or weight.dim() != 1):
            raise ValueError("weight must be a 1-D tensor with one element per class")
        self.register_buffer("weight", weight)
        self.weight: Optional[torch.Tensor]
        self.ignore_index = int(ignore_index)
        self.reduction = reduction
        self.label_smoothing = label_smoothing

    def extra_repr(self) -> str:
        return f"ignore_index={self.ignore_index}, reduction={self.reduction!r}, label_smoothing={self.label_smoothing}"

    def _is_default(self, targets: torch.Tensor) -> bool:
        return (self.weight is None and self.ignore_index == -100 and self.reduction == "mean"
                and self.label_smoothing == 0.0 and targets.dtype == torch.int64)

    def forward(self, outputs: torch.Tensor, targets: torch.Tensor) -> torch.Tensor:
        if not outputs.is_cuda:
            raise RuntimeError("b200seg.CrossEntropyLoss runs on CUDA only (no CPU fallback)")
        if outputs.dim() != 4:
            raise ValueError("expected NCHW logits")
        if self._is_default(targets):
            return _FusedCE.apply(outputs.float(), targets)
        if targets.dtype not in (torch.int64, torch.uint8):
            raise TypeError(f"b200seg.CrossEntropyLoss: targets must be int64 or uint8 class indices, got {targets.dtype}")
        B, C, H, W = outputs.shape
        if tuple(targets.shape) != (B, H, W):
            raise ValueError(f"targets {tuple(targets.shape)} do not match logits {tuple(outputs.shape)}: expected {(B, H, W)}")
        weight = self.weight
        if weight is not None:
            if weight.numel() != C:
                raise RuntimeError(f"weight tensor should be defined either for all {C} classes or no classes but got "
                                   f"weight tensor of shape: {list(weight.shape)}")
            weight = weight.float().contiguous()
        return _FusedCEEx.apply(outputs.float(), targets, weight, self.ignore_index, self.label_smoothing, self.reduction)


def _legacy_reduction(size_average, reduce) -> str:
    """torch's mapping of the deprecated arguments (torch.nn._reduction.legacy_get_string), with its warning."""
    size_average = True if size_average is None else size_average
    reduce = True if reduce is None else reduce
    ret = "none" if not reduce else ("mean" if size_average else "sum")
    warnings.warn(f"size_average and reduce args will be deprecated, please use reduction='{ret}' instead.")
    return ret
