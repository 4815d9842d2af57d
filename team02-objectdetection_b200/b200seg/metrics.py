"""Validation metrics for semantic segmentation, accumulated on the GPU.

The reference's validation loop (train.py:46-74) is commented out, so its "best validation loss" is always inf.  This is
what that loop would compute -- mean cross-entropy -- plus the confusion matrix and what follows from it (pixel accuracy,
per-class IoU, mIoU):

    metrics = b200seg.SegmentationMetrics(num_classes=10)
    model.eval()
    for x, t in val_loader:
        model.evaluate(x, t, metrics)       # MobileNetV2UNet in bf16: the metrics are taken inside the output-tail kernel
    metrics.update(logits, t)               # any NCHW f32 / bf16 logits
    res = metrics.compute()                 # one device-to-host copy

``update`` and ``evaluate`` never synchronise with the host: they enqueue kernels on the current stream and can be
captured in a CUDA graph.  The state stays on the device until ``compute``.
"""
from __future__ import annotations

import torch

from . import ops

MAX_CLASSES = 64          # the standalone kernel keeps a [C][C] u32 histogram per CTA in shared memory (16 KB at 64)


class SegmentationMetrics:
    """Device-side accumulator of the confusion matrix (rows = targets, columns = predictions; the argmax over classes,
    first maximum wins as in ``torch.argmax``), the number of ``valid`` pixels (target in [0, C)), of ``invalid`` ones
    (neither in range nor ``ignore_index``) and the f64 sum of the per-pixel cross-entropy over the valid pixels.

    Targets are int64 (``CrossEntropyLoss`` targets) or uint8 label maps; the same ``ignore_index`` rule applies to both,
    so a uint8 map marks ignored pixels with e.g. ``ignore_index=255``.  Pixels whose target equals ``ignore_index``
    contribute nothing, also when it is a class index (``ignore_index=0`` drops class 0 from the loss, the counts and the
    confusion matrix, like ``nn.CrossEntropyLoss(ignore_index=0)``)."""

    def __init__(self, num_classes: int, device="cuda", ignore_index: int = ops.IGNORE_INDEX):
        if not 1 <= int(num_classes) <= MAX_CLASSES:
            raise ValueError(f"num_classes must be in [1, {MAX_CLASSES}], got {num_classes}")
        self.num_classes = int(num_classes)
        self.ignore_index = int(ignore_index)
        C = self.num_classes
        # ONE int64 buffer: [C*C confusion | valid | invalid | loss_sum (f64 bits)]: one memset to reset, one copy to read
        self._buf = torch.zeros(C * C + 3, dtype=torch.int64, device=device)
        self.confusion = self._buf[:C * C].view(C, C)
        self.counts = self._buf[C * C:C * C + 2]
        self.loss_sum = self._buf[C * C + 2:].view(torch.float64)

    @property
    def device(self) -> torch.device:
        return self._buf.device

    def reset(self) -> "SegmentationMetrics":
        self._buf.zero_()
        return self

    def _check(self, x: torch.Tensor, target: torch.Tensor):
        if not x.is_cuda or not target.is_cuda or not self._buf.is_cuda:
            raise RuntimeError("SegmentationMetrics runs on CUDA tensors only (no CPU fallback)")
        if x.device != self.device or target.device != self.device:
            raise ValueError(f"inputs on {x.device} / {target.device} but the metrics state is on {self.device}")
        if target.dtype not in (torch.int64, torch.uint8):
            raise ValueError(f"targets must be int64 or uint8, got {target.dtype}")
        if target.dim() != 3 or target.shape[0] != x.shape[0] or tuple(target.shape[1:]) != tuple(x.shape[2:]):
            raise ValueError(f"target shape {tuple(target.shape)} is not [B,H,W] of the input {tuple(x.shape)}")

    def update(self, logits: torch.Tensor, target: torch.Tensor) -> "SegmentationMetrics":
        """Accumulate the metrics of NCHW f32 / bf16 ``logits`` [B,C,H,W] against ``target`` [B,H,W]."""
        if logits.dim() != 4:
            raise ValueError(f"logits must be NCHW [B,C,H,W], got {tuple(logits.shape)}")
        self._check(logits, target)
        if logits.shape[1] != self.num_classes:
            raise ValueError(f"logits have {logits.shape[1]} classes, the metrics {self.num_classes}")
        if logits.dtype not in (torch.float32, torch.bfloat16):
            raise ValueError(f"logits must be float32 or bfloat16, got {logits.dtype}")
        with torch.cuda.device(logits.device):
            ops.seg_metrics(logits.contiguous(), target, self.num_classes, self.ignore_index, self.confusion, self.counts,
                            self.loss_sum)
        return self

    def all_reduce(self, group=None) -> "SegmentationMetrics":
        """Data-parallel validation: sum the state over the ranks of ``group`` with ONE collective.  The counts travel as
        f64 (exact below 2^53 pixels) packed with the loss sum."""
        import torch.distributed as dist
        C = self.num_classes
        packed = torch.cat([self._buf[:C * C + 2].to(torch.float64), self.loss_sum])
        dist.all_reduce(packed, op=dist.ReduceOp.SUM, group=group)
        self._buf[:C * C + 2].copy_(packed[:C * C + 2].round().to(torch.int64))
        self.loss_sum.copy_(packed[C * C + 2:])
        return self

    def compute(self) -> dict:
        """Host-side results (one device-to-host copy):
        ``loss`` = loss_sum / valid (NaN if invalid > 0 or valid == 0, the policy of b200seg.CrossEntropyLoss),
        ``pixel_accuracy`` = trace / valid, ``iou`` f64 [C] = cm[c,c] / (row_c + col_c - cm[c,c]) (NaN for a class absent
        from both targets and predictions), ``miou`` = NaN-mean of ``iou``, and ``confusion``, ``valid``, ``invalid``."""
        C = self.num_classes
        buf = self._buf.cpu()
        cm = buf[:C * C].view(C, C).clone()
        valid, invalid = int(buf[C * C]), int(buf[C * C + 1])
        loss_sum = float(buf[C * C + 2:].view(torch.float64)[0])
        nan = float("nan")
        cmd = cm.to(torch.float64)
        tp = cmd.diagonal()
        union = cmd.sum(1) + cmd.sum(0) - tp
        iou = torch.where(union > 0, tp / union.clamp_min(1), torch.full_like(tp, nan))
        present = ~torch.isnan(iou)
        return {
            "loss": loss_sum / valid if valid > 0 and invalid == 0 else nan,
            "pixel_accuracy": float(tp.sum()) / valid if valid > 0 else nan,
            "iou": iou,
            "miou": float(iou[present].mean()) if bool(present.any()) else nan,
            "confusion": cm,
            "valid": valid,
            "invalid": invalid,
        }

    def __repr__(self):
        return f"SegmentationMetrics(num_classes={self.num_classes}, device={self.device}, ignore_index={self.ignore_index})"
