"""Drop-in `nn.Module`s for the reference's segmentation models, computed by sm_100a kernels.

Mirrors /root/reference/src/unet.py:
  * ``MobileNetV2UNet(output_channels=1)``            unet.py:7-51
  * ``UNet(output_channels=1, base_filters=64)``      unet.py:124-147
  * ``LightUNet(base_filters=32)``                    unet.py:149-172
and the blocks ``double_conv / inconv / down / up / outconv`` (unet.py:53-121).

What is kept identical (SURVEY.md §8b, Appendix A): constructor signatures, attribute names,
child registration order, the 691-key aliased ``state_dict`` (``downK.N.*`` shares storage with
``backbone.features.N.*``; the unused ``backbone.classifier`` is present), ``named_parameters()``
order, ``forward(x) -> logits`` in NCHW.

What is different: the child modules are *parameter containers only*.  ``forward`` hands the
whole network to ``b200seg.engine`` which runs hand-written CUDA kernels through the C-ABI in
``libb200seg.so``.  There is no CPU / eager fallback: a CPU tensor or a missing library raises.

The encoder topology restates torchvision 0.26 ``models/mobilenetv2.py:19-64,101-161`` (the
reference depends on it un-vendored, requirements.txt:2); torchvision itself is NOT imported.
"""
from __future__ import annotations

import math
from typing import List, Optional

import torch
import torch.nn as nn

# torchvision mobilenetv2.py:105-114  (t, c, n, s)
_MBV2_SETTING = [(1, 16, 1, 1), (6, 24, 2, 2), (6, 32, 3, 2), (6, 64, 4, 2),
                 (6, 96, 3, 1), (6, 160, 3, 2), (6, 320, 1, 1)]


def _container_forward(self, *a, **k):  # pragma: no cover - guard
    raise RuntimeError(
        f"{type(self).__name__} is a parameter container of the B200 drop-in; call the top-level "
        "model (MobileNetV2UNet / UNet), which runs the fused CUDA path. There is no eager fallback.")


class ConvBNAct(nn.Sequential):
    """Container with torchvision ``Conv2dNormActivation``'s child layout (ops/misc.py:86-116):
    '0' Conv2d(bias=False), '1' BatchNorm2d, '2' ReLU6."""

    def __init__(self, cin, cout, kernel_size=3, stride=1, groups=1):
        pad = (kernel_size - 1) // 2
        super().__init__(nn.Conv2d(cin, cout, kernel_size, stride, pad, groups=groups, bias=False),
                         nn.BatchNorm2d(cout), nn.ReLU6(inplace=True))
        self.out_channels = cout

    forward = _container_forward


class InvertedResidual(nn.Module):
    """Container with torchvision ``InvertedResidual``'s child layout (mobilenetv2.py:19-64)."""

    def __init__(self, inp, oup, stride, expand_ratio):
        super().__init__()
        self.stride = stride
        hidden = int(round(inp * expand_ratio))
        self.use_res_connect = stride == 1 and inp == oup
        layers: List[nn.Module] = []
        if expand_ratio != 1:
            layers.append(ConvBNAct(inp, hidden, kernel_size=1))
        layers += [ConvBNAct(hidden, hidden, stride=stride, groups=hidden),
                   nn.Conv2d(hidden, oup, 1, 1, 0, bias=False), nn.BatchNorm2d(oup)]
        self.conv = nn.Sequential(*layers)
        self.inp, self.oup, self.hidden, self.expand_ratio = inp, oup, hidden, expand_ratio
        self.out_channels = oup

    forward = _container_forward


class MobileNetV2(nn.Module):
    """Encoder container: ``features`` (19 children) + the never-used ``classifier``
    (mobilenetv2.py:101-161; SURVEY finding 5: classifier stays in parameters()/state_dict)."""

    def __init__(self, num_classes=1000, dropout=0.2):
        super().__init__()
        feats: List[nn.Module] = [ConvBNAct(3, 32, stride=2)]
        inp = 32
        for t, c, n, s in _MBV2_SETTING:
            for i in range(n):
                feats.append(InvertedResidual(inp, c, s if i == 0 else 1, t))
                inp = c
        feats.append(ConvBNAct(inp, 1280, kernel_size=1))
        self.features = nn.Sequential(*feats)
        self.classifier = nn.Sequential(nn.Dropout(p=dropout), nn.Linear(1280, num_classes))
        # init: mobilenetv2.py:151-161
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out")
            elif isinstance(m, nn.BatchNorm2d):
                nn.init.ones_(m.weight); nn.init.zeros_(m.bias)
            elif isinstance(m, nn.Linear):
                nn.init.normal_(m.weight, 0, 0.01); nn.init.zeros_(m.bias)

    forward = _container_forward


class double_conv(nn.Module):
    """(conv3x3+bias => BN => ReLU) * 2 -- unet.py:53-68 (container)."""

    def __init__(self, in_ch, out_ch):
        super().__init__()
        self.conv = nn.Sequential(
            nn.Conv2d(in_ch, out_ch, 3, padding=1), nn.BatchNorm2d(out_ch), nn.ReLU(inplace=True),
            nn.Conv2d(out_ch, out_ch, 3, padding=1), nn.BatchNorm2d(out_ch), nn.ReLU(inplace=True))

    forward = _container_forward


class inconv(nn.Module):
    """unet.py:71-78."""

    def __init__(self, in_ch, out_ch):
        super().__init__()
        self.conv = double_conv(in_ch, out_ch)

    forward = _container_forward


class down(nn.Module):
    """MaxPool2d(2) + double_conv -- unet.py:81-91."""

    def __init__(self, in_ch, out_ch):
        super().__init__()
        self.mpconv = nn.Sequential(nn.MaxPool2d(2), double_conv(in_ch, out_ch))

    forward = _container_forward


class up(nn.Module):
    """bilinear x2 (align_corners=False) + cat([skip, up]) + double_conv -- unet.py:94-105."""

    def __init__(self, in_ch, out_ch):
        super().__init__()
        self.up = nn.Upsample(scale_factor=2, mode="bilinear")
        self.conv = double_conv(in_ch, out_ch)

    forward = _container_forward


class outconv(nn.Module):
    """1x1+b => BN => ReLU => 1x1+b -- unet.py:108-121."""

    def __init__(self, in_ch, out_ch):
        super().__init__()
        self.conv = nn.Sequential(nn.Conv2d(in_ch, in_ch // 2, 1), nn.BatchNorm2d(in_ch // 2),
                                  nn.ReLU(inplace=True), nn.Conv2d(in_ch // 2, out_ch, 1))

    forward = _container_forward


class _EngineModel(nn.Module):
    """Shared plumbing: lazily builds the CUDA engine and routes forward through it."""

    _arch = ""

    def _get_engine(self):
        eng = self.__dict__.get("_engine")
        if eng is None:
            from . import engine  # imports the C-ABI library; raises loudly if it is missing
            eng = engine.Engine(self, self._arch)
            self.__dict__["_engine"] = eng      # not a submodule / not in state_dict
        return eng

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if not x.is_cuda:
            raise RuntimeError("b200seg models run on CUDA (sm_100a) only; got a CPU tensor. "
                               "There is deliberately no CPU fallback.")
        return self._get_engine().forward(x)

    @torch.no_grad()
    def predict_mask(self, x: torch.Tensor, out: torch.Tensor = None) -> torch.Tensor:
        """Fused final-upsample + argmax -> uint8 class mask [B,H,W] (what inference.py:64-65
        computes on the host from the logits).  Eval mode only.  ``out``: an existing uint8 [B,H,W] tensor to write
        (a frame loop that hands the mask to another stream keeps two of them instead of allocating per frame)."""
        return self._get_engine().forward(x, want_mask=True, out=out)

    @torch.no_grad()
    def evaluate(self, x: torch.Tensor, target: torch.Tensor, metrics):
        """Validation step (the reference's commented-out loop, train.py:46-74): the forward of ``x`` with the loss,
        argmax and confusion histogram against ``target`` (int64 [B,H,W] CrossEntropyLoss targets, or uint8) accumulated
        into ``metrics`` (b200seg.SegmentationMetrics) on the device.  No logits tensor is returned (MobileNetV2UNet in
        bf16 never writes one: the output-tail kernel takes the metrics itself).  Eval mode only; never synchronises
        with the host.  Returns ``metrics``."""
        if self.training:
            raise RuntimeError("evaluate needs model.eval()")
        if not x.is_cuda:
            raise RuntimeError("b200seg models run on CUDA (sm_100a) only; got a CPU tensor. "
                               "There is deliberately no CPU fallback.")
        if metrics.num_classes != self.output_channels:
            raise ValueError(f"metrics count {metrics.num_classes} classes, the model outputs {self.output_channels}")
        metrics._check(x, target)
        self._get_engine().forward(x, metrics=(metrics, target))
        return metrics


class MobileNetV2UNet(_EngineModel):
    """unet.py:7-51.  NOTE unet.py:12 downloads ImageNet weights; offline that is impossible, so
    the encoder is random-initialised exactly like ``mobilenet_v2(weights=None)``.  Load a
    reference checkpoint with ``load_state_dict`` (691 keys, strict) to get trained weights."""

    _arch = "mbv2unet"

    def __init__(self, output_channels=1):
        super().__init__()
        self.backbone = MobileNetV2()
        self.down1 = self.backbone.features[:2]      # unet.py:15-19: aliasing slices (index kept)
        self.down2 = self.backbone.features[2:4]
        self.down3 = self.backbone.features[4:7]
        self.down4 = self.backbone.features[7:11]
        self.down5 = self.backbone.features[11:19]
        self.up1 = up(1280 + 64, 256)
        self.up2 = up(256 + 32, 128)
        self.up3 = up(128 + 24, 64)
        self.up4 = up(64 + 16, 32)
        self.outc = outconv(32, output_channels)
        self.final_upsample = nn.Upsample(scale_factor=2, mode="bilinear", align_corners=True)
        self.output_channels = output_channels


class UNet(_EngineModel):
    """unet.py:124-147."""

    _arch = "unet"

    def __init__(self, output_channels=1, base_filters=64):
        super().__init__()
        b = base_filters
        self.inc = inconv(3, b)
        self.down1 = down(b, b * 2)
        self.down2 = down(b * 2, b * 4)
        self.down3 = down(b * 4, b * 4)
        self.up1 = up(b * 8, b * 2)
        self.up2 = up(b * 4, b)
        self.up3 = up(b * 2, b)
        self.sem_out = outconv(b, output_channels)
        self.output_channels = output_channels
        self.base_filters = b


class LightUNet(UNet):
    """unet.py:149-172: UNet with base 32 and a single output channel."""

    def __init__(self, base_filters=32):
        super().__init__(output_channels=1, base_filters=base_filters)
