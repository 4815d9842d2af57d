"""Tensor-level wrappers over the C ABI: one function per ATen dispatch of the reference hot path
(SURVEY.md section 2.1).  Each validates device/dtype/layout, passes raw pointers and the current
CUDA stream, and returns the output tensor.  Activations are NHWC-contiguous torch tensors of shape
[B, H, W, C]; nothing here ever falls back to torch arithmetic.
"""
from __future__ import annotations

from typing import Optional

import os

import torch

from . import _cabi
from ._cabi import ACT_NONE, ACT_RELU, ACT_RELU6, BF16, F32, check, lib, ptr  # noqa: F401

_DT = {torch.float32: F32, torch.bfloat16: BF16}


def _dt(t: torch.Tensor) -> int:
    try:
        return _DT[t.dtype]
    except KeyError:
        raise TypeError(f"b200seg supports float32 and bfloat16 activations, got {t.dtype}") from None


def _cuda(*ts):
    for t in ts:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("b200seg ops need CUDA tensors (no CPU fallback)")
        if not t.is_contiguous():
            raise RuntimeError("b200seg ops need contiguous tensors")


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


_MUTATION_EPOCH = 0


def mutation_epoch() -> int:
    return _MUTATION_EPOCH


def bump_mutation_epoch() -> None:
    """Called by every code path that writes parameters or BatchNorm buffers through raw device pointers (fused Adam,
    the training forward, CUDA-graph replays of it): tensor._version does not see those writes, and the eval-mode
    packed-weight cache must."""
    global _MUTATION_EPOCH
    _MUTATION_EPOCH += 1


def conv3x3_smallcin(x_nchw, w, b, stride: int, act: int, out_dtype, out=None):
    """x NCHW [B,Cin<=4,H,W]; w f32 [3,3,Cin,Cout]; -> NHWC [B,Ho,Wo,Cout]."""
    _cuda(x_nchw, w, b)
    B, Cin, H, W = x_nchw.shape
    Cout = w.shape[-1]
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    if out is None:
        out = torch.empty((B, Ho, Wo, Cout), device=x_nchw.device, dtype=out_dtype)
    check(lib.b200seg_conv3x3_smallcin(ptr(x_nchw), _dt(x_nchw), ptr(w), ptr(b), ptr(out), _dt(out), B, Cin, H, W,
                                       Cout, stride, act, _stream()), "conv3x3_smallcin")
    return out


def stem_mb1_supported(x_nchw, cstem: int, cout: int) -> bool:
    return bool(lib.b200seg_stem_mb1_supported(_dt(x_nchw), x_nchw.shape[2], x_nchw.shape[3], cstem, cout))


def stem_mb1(x_nchw, w_stem, b_stem, w_dw, b_dw, w_pw, b_pw, out=None):
    """features.0 + features.1 in one kernel: NCHW f32 frames -> NHWC bf16 [B,H/2,W/2,16] (csrc/stem_mb1.cu)."""
    _cuda(x_nchw, w_stem, b_stem, w_dw, b_dw, w_pw, b_pw)
    B, C, H, W = x_nchw.shape
    if C != 3 or not x_nchw.is_contiguous():
        raise ValueError("stem_mb1 expects a contiguous NCHW tensor with 3 channels")
    if w_dw.dtype != torch.bfloat16 or w_pw.dtype != torch.bfloat16 or w_stem.dtype != torch.float32:
        raise TypeError("stem_mb1: w_stem f32, w_dw / w_pw bf16")
    if out is None:
        out = torch.empty((B, H // 2, W // 2, w_pw.shape[0]), device=x_nchw.device, dtype=torch.bfloat16)
    check(lib.b200seg_stem_mb1(ptr(x_nchw), _dt(x_nchw), ptr(w_stem), ptr(b_stem), ptr(w_dw), ptr(b_dw), ptr(w_pw), ptr(b_pw),
                               ptr(out), B, H, W, _stream()), "stem_mb1")
    return out


def dwconv3x3(x, w9c, b, stride: int, act: int, out=None):
    """x NHWC; w9c f32 [9,C]."""
    _cuda(x, w9c, b)
    B, H, W, Cc = x.shape
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    if out is None:
        out = torch.empty((B, Ho, Wo, Cc), device=x.device, dtype=x.dtype)
    check(lib.b200seg_dwconv3x3(ptr(x), ptr(w9c), ptr(b), ptr(out), _dt(x), B, H, W, Cc, stride, act, _stream()),
          "dwconv3x3")
    return out


def dwconv3x3_bf16w(x, w9c_bf16, b, stride: int, act: int, out=None, variant: int = 0):
    """Depthwise 3x3 on bf16 activations with bf16 taps [9,C] (mixed-precision FMA, no unpack instructions)."""
    _cuda(x, w9c_bf16, b)
    if x.dtype != torch.bfloat16 or w9c_bf16.dtype != torch.bfloat16:
        raise TypeError("dwconv3x3_bf16w is bf16-only")
    B, H, W, Cc = x.shape
    if tuple(w9c_bf16.shape) != (9, Cc):
        raise ValueError(f"dwconv3x3_bf16w: taps {tuple(w9c_bf16.shape)} != (9, {Cc})")
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    if out is None:
        out = torch.empty((B, Ho, Wo, Cc), device=x.device, dtype=torch.bfloat16)
    check(lib.b200seg_dwconv3x3_bf16w(ptr(x), ptr(w9c_bf16), ptr(b), ptr(out), B, H, W, Cc, stride, act, variant, _stream()),
          "dwconv3x3_bf16w")
    return out


def pack_dw_diag(w9c: torch.Tensor) -> torch.Tensor:
    """f32 [9, C] depthwise taps -> block-diagonal bf16 [C, 9, 64] for dwconv3x3_tc."""
    C = w9c.shape[1]
    out = torch.zeros(C, 9, 64, device=w9c.device, dtype=torch.bfloat16)
    idx = torch.arange(C, device=w9c.device)
    out[idx, :, idx % 64] = w9c.t().to(torch.bfloat16)
    return out.contiguous()


def dwconv3x3_tc(x, wdiag, b, stride: int, act: int, out=None, flags: int = 0):
    """Depthwise 3x3 on the tensor cores. x NHWC bf16; wdiag from pack_dw_diag."""
    _cuda(x, wdiag, b)
    if x.dtype != torch.bfloat16 or wdiag.dtype != torch.bfloat16:
        raise TypeError("dwconv3x3_tc is bf16-only")
    B, H, W, Cc = x.shape
    if tuple(wdiag.shape) != (Cc, 9, 64):
        raise ValueError(f"dwconv3x3_tc: wdiag {tuple(wdiag.shape)} != ({Cc}, 9, 64)")
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    if out is None:
        out = torch.empty((B, Ho, Wo, Cc), device=x.device, dtype=torch.bfloat16)
    check(lib.b200seg_dwconv3x3_tc(ptr(x), ptr(wdiag), ptr(b), ptr(out), B, H, W, Cc, stride, act, flags, _stream()),
          "dwconv3x3_tc")
    return out


USE_CONV_RS = True       # 3x3 convs with <= 32 output channels on wide maps go through the row-stacked kernel (conv_rs.cu)
CONV_RS_FLAGS = 0        # tuning flags of b200seg_conv_rs (tools only)


def conv_rs(x, w, b, act: int, res=None, out=None, flags: int = 0):
    """Row-stacked 3x3 tensor-core conv for few output channels: same operands/results as conv_tc(taps=9)."""
    _cuda(x, w, b, res)
    if x.dtype != torch.bfloat16 or w.dtype != torch.bfloat16:
        raise TypeError("conv_rs is bf16-only")
    B, H, W, Cin = x.shape
    Cout = w.shape[0]
    if w.shape[1] != 9 * Cin:
        raise ValueError(f"conv_rs: weight {tuple(w.shape)} does not match Cin={Cin}")
    if out is None:
        out = torch.empty((B, H, W, Cout), device=x.device, dtype=torch.bfloat16)
    check(lib.b200seg_conv_rs(ptr(x), ptr(w), ptr(b), ptr(res), ptr(out), B, H, W, Cin, Cout, act, flags, _stream()), "conv_rs")
    return out


def conv_tc(x, w, b, taps: int, act: int, res=None, out=None, flags: int = 0):
    """Tensor-core conv. x NHWC bf16 [B,H,W,Cin]; w bf16 [Cout, taps*Cin]; b f32 [Cout]."""
    _cuda(x, w, b, res)
    if x.dtype != torch.bfloat16 or w.dtype != torch.bfloat16:
        raise TypeError("conv_tc is bf16-only")
    B, H, W, Cin = x.shape
    Cout = w.shape[0]
    if w.shape[1] != taps * Cin:
        raise ValueError(f"conv_tc: weight {tuple(w.shape)} does not match taps={taps} Cin={Cin}")
    # the 80-column variant (data gradient of up4.conv.0) only without a residual: its per-pixel epilogue reads a 160-byte
    # residual row in ten 16-byte pieces with 255 registers live (203 us against conv_tc's 167; 93 against 144 without)
    if (taps == 9 and USE_CONV_RS and flags == 0 and lib.b200seg_conv_rs_supported(H, W, Cin, Cout)
            and (Cout <= 32 or res is None)):
        return conv_rs(x, w, b, act, res, out, CONV_RS_FLAGS)
    if out is None:
        out = torch.empty((B, H, W, Cout), device=x.device, dtype=torch.bfloat16)
    check(lib.b200seg_conv_tc(ptr(x), ptr(w), ptr(b), ptr(res), ptr(out), B, H, W, Cin, Cout, taps, act, flags,
                              _stream()), "conv_tc")
    return out


def conv_simt(x, w, b, taps: int, act: int, res=None, out=None):
    """FP32-pipe conv. x NHWC (f32|bf16); w f32 [Cout, taps*Cin]."""
    _cuda(x, w, b, res)
    if w.dtype != torch.float32:
        raise TypeError("conv_simt weights are f32")
    B, H, W, Cin = x.shape
    Cout = w.shape[0]
    if w.shape[1] != taps * Cin:
        raise ValueError(f"conv_simt: weight {tuple(w.shape)} does not match taps={taps} Cin={Cin}")
    if out is None:
        out = torch.empty((B, H, W, Cout), device=x.device, dtype=x.dtype)
    check(lib.b200seg_conv_simt(ptr(x), ptr(w), ptr(b), ptr(res), ptr(out), _dt(x), B, H, W, Cin, Cout, taps, act,
                                _stream()), "conv_simt")
    return out


def pad_channels(t: torch.Tensor, mult: int) -> torch.Tensor:
    """Zero-pad the LAST dim of a parameter vector/matrix to a multiple of `mult` (fused-block operand layout)."""
    c = t.shape[-1]
    cp = (c + mult - 1) // mult * mult
    if cp == c:
        return t.contiguous()
    out = torch.zeros((*t.shape[:-1], cp), device=t.device, dtype=t.dtype)
    out[..., :c] = t
    return out


def mbconv(x, w_exp, b_exp, w_dw, b_dw, w_proj, b_proj, stride: int, residual: bool, out=None, flags: int = 0):
    """Fused inverted-residual block (expand 1x1 + ReLU6 -> depthwise 3x3 + ReLU6 -> project 1x1 [+ x]), bf16 NHWC.
    w_exp [Ce, Cin] bf16, w_proj [Cout, Ce] bf16; b_exp/b_dw f32 [ceil64(Ce)], w_dw bf16 [9, ceil64(Ce)],
    b_proj f32 [ceil16(Cout)] (see pad_channels)."""
    _cuda(x, w_exp, b_exp, w_dw, b_dw, w_proj, b_proj)
    if x.dtype != torch.bfloat16 or w_exp.dtype != torch.bfloat16 or w_proj.dtype != torch.bfloat16 or w_dw.dtype != torch.bfloat16:
        raise TypeError("mbconv is bf16-only (activations, 1x1 weights and depthwise taps)")
    B, H, W, Cin = x.shape
    Ce, Cout = w_exp.shape[0], w_proj.shape[0]
    cep, cop = (Ce + 63) // 64 * 64, (Cout + 15) // 16 * 16
    if (tuple(w_exp.shape) != (Ce, Cin) or tuple(w_proj.shape) != (Cout, Ce) or tuple(w_dw.shape) != (9, cep)
            or b_exp.numel() != cep or b_dw.numel() != cep or b_proj.numel() != cop):
        raise ValueError(f"mbconv: operand shapes w_exp {tuple(w_exp.shape)} w_dw {tuple(w_dw.shape)} "
                         f"w_proj {tuple(w_proj.shape)} b {b_exp.numel()},{b_dw.numel()},{b_proj.numel()}")
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    if out is None:
        out = torch.empty((B, Ho, Wo, Cout), device=x.device, dtype=torch.bfloat16)
    check(lib.b200seg_mbconv(ptr(x), ptr(w_exp), ptr(b_exp), ptr(w_dw), ptr(b_dw), ptr(w_proj), ptr(b_proj),
                             1 if residual else 0, ptr(out), B, H, W, Cin, Ce, Cout, stride, flags, _stream()), "mbconv")
    return out


def upsample2x_concat(skip, x, out=None):
    """cat([skip, bilinear_x2(x, align_corners=False)], channel) in NHWC."""
    _cuda(skip, x)
    B, h, w, Cu = x.shape
    Cs = skip.shape[3]
    if skip.shape[:3] != (B, 2 * h, 2 * w) or skip.dtype != x.dtype:
        raise ValueError(f"upsample2x_concat: skip {tuple(skip.shape)} vs x {tuple(x.shape)}")
    if out is None:
        out = torch.empty((B, 2 * h, 2 * w, Cs + Cu), device=x.device, dtype=x.dtype)
    check(lib.b200seg_upsample2x_concat(ptr(skip), ptr(x), ptr(out), _dt(x), B, h, w, Cs, Cu, _stream()),
          "upsample2x_concat")
    return out


def upsample2x_ac_nchw(logits, C: int, out_dtype, out=None):
    """NHWC logits [B,h,w,ldc] -> NCHW [B,C,2h,2w], bilinear align_corners=True."""
    _cuda(logits)
    B, h, w, ldc = logits.shape
    if out is None:
        out = torch.empty((B, C, 2 * h, 2 * w), device=logits.device, dtype=out_dtype)
    if ldc != 16:           # more than 16 classes: generic kernel (csrc/generic_ops.cu)
        check(lib.b200seg_upsample2x_ac_generic(ptr(logits), _dt(logits), ldc, ptr(out), _dt(out), None, B, h, w, C,
                                                _stream()), "upsample2x_ac_generic")
        return out
    check(lib.b200seg_upsample2x_ac_nchw(ptr(logits), _dt(logits), ldc, ptr(out), _dt(out), B, h, w, C, _stream()),
          "upsample2x_ac_nchw")
    return out


def upsample2x_ac_argmax(logits, C: int, out=None):
    _cuda(logits)
    B, h, w, ldc = logits.shape
    if out is None:
        out = torch.empty((B, 2 * h, 2 * w), device=logits.device, dtype=torch.uint8)
    if ldc != 16:
        check(lib.b200seg_upsample2x_ac_generic(ptr(logits), _dt(logits), ldc, None, F32, ptr(out), B, h, w, C,
                                                _stream()), "upsample2x_ac_generic")
        return out
    check(lib.b200seg_upsample2x_ac_argmax(ptr(logits), _dt(logits), ldc, ptr(out), B, h, w, C, _stream()),
          "upsample2x_ac_argmax")
    return out


def tail_fused(x, w0, b0, w3, b3, C: int, out_dtype=None, want_mask: bool = False, out=None):
    """outconv(32, C) + final_upsample (+ argmax) in one kernel.  x NHWC bf16 [B,h,w,32]; w0 bf16 [16,32], b0 f32 [>=16];
    w3 bf16 [16,16], b3 f32 [>=16].  Returns NCHW [B,C,2h,2w] of out_dtype, or the uint8 mask [B,2h,2w]."""
    _cuda(x, w0, b0, w3, b3)
    B, h, w, cin = x.shape
    if (x.dtype != torch.bfloat16 or cin != 32 or tuple(w0.shape) != (16, 32) or tuple(w3.shape) != (16, 16)
            or w0.dtype != torch.bfloat16 or w3.dtype != torch.bfloat16 or b0.numel() < 16 or b3.numel() < 16 or not 1 <= C <= 16):
        raise ValueError("tail_fused: expects the MobileNetV2UNet tail (32 -> 16 -> C <= 16 channels, bf16)")
    if out is not None:
        want = (B, 2 * h, 2 * w) if want_mask else (B, C, 2 * h, 2 * w)
        if (tuple(out.shape) != want or out.dtype != (torch.uint8 if want_mask else out_dtype) or not out.is_contiguous()
                or out.device != x.device):
            raise ValueError(f"tail_fused: out must be a contiguous {want} tensor of the result dtype on {x.device}")
    if want_mask:
        if out is None:
            out = torch.empty((B, 2 * h, 2 * w), device=x.device, dtype=torch.uint8)
        check(lib.b200seg_tail_fused(ptr(x), ptr(w0), ptr(b0), ptr(w3), ptr(b3), None, F32, ptr(out), B, h, w, C, _stream()),
              "tail_fused")
    else:
        if out is None:
            out = torch.empty((B, C, 2 * h, 2 * w), device=x.device, dtype=out_dtype)
        check(lib.b200seg_tail_fused(ptr(x), ptr(w0), ptr(b0), ptr(w3), ptr(b3), ptr(out), _dt(out), None, B, h, w, C, _stream()),
              "tail_fused")
    return out


_TGT = {torch.int64: _cabi.I64, torch.uint8: _cabi.U8}


def _metrics_target(target, shape):
    """int64 | uint8 label map of ``shape``, contiguous and 16-byte aligned for the kernels' vector loads: a non-contiguous
    or misaligned view (a crop of a larger label map) is copied."""
    if target.dtype not in _TGT:
        raise ValueError(f"targets must be int64 or uint8, got {target.dtype}")
    if tuple(target.shape) != tuple(shape):
        raise ValueError(f"target shape {tuple(target.shape)} does not match the logits' [B,H,W] {tuple(shape)}")
    target = target.contiguous()
    if target.data_ptr() % 16:                   # a view at an odd offset: the 16-byte target loads need an aligned copy
        target = target.clone()
    return target


def tail_fused_metrics(x, w0, b0, w3, b3, C: int, target, ignore_index: int, confusion, counts, loss_sum):
    """outconv(32, C) + final_upsample + validation metrics in one kernel (operands as tail_fused): adds the confusion
    matrix, [valid, invalid] counts and the cross-entropy sum of ``target`` [B,2h,2w] into the int64 / f64 state."""
    _cuda(x, w0, b0, w3, b3, confusion, counts, loss_sum)
    B, h, w, cin = x.shape
    if (x.dtype != torch.bfloat16 or cin != 32 or tuple(w0.shape) != (16, 32) or tuple(w3.shape) != (16, 16)
            or w0.dtype != torch.bfloat16 or w3.dtype != torch.bfloat16 or b0.numel() < 16 or b3.numel() < 16 or not 1 <= C <= 16):
        raise ValueError("tail_fused_metrics: expects the MobileNetV2UNet tail (32 -> 16 -> C <= 16 channels, bf16)")
    target = _metrics_target(target, (B, 2 * h, 2 * w))
    _cuda(target)
    check(lib.b200seg_tail_fused_metrics(ptr(x), ptr(w0), ptr(b0), ptr(w3), ptr(b3), ptr(target), _TGT[target.dtype],
                                         int(ignore_index), ptr(confusion), ptr(counts), ptr(loss_sum), B, h, w, C, _stream()),
          "tail_fused_metrics")


def seg_metrics(logits, target, C: int, ignore_index: int, confusion, counts, loss_sum, nhwc: bool = False):
    """Validation metrics over existing logits: NCHW [B,C,H,W] (``nhwc`` False) or NHWC [B,H,W,ldc >= C] (f32 | bf16),
    int64 | uint8 targets [B,H,W]; adds into the int64 / f64 state like tail_fused_metrics."""
    _cuda(logits, confusion, counts, loss_sum)
    if logits.dim() != 4:
        raise ValueError(f"logits must be 4-D, got {tuple(logits.shape)}")
    if nhwc:
        B, H, W, ldc = logits.shape
    else:
        B, Cl, H, W = logits.shape
        ldc = 0
        if Cl != C:
            raise ValueError(f"logits have {Cl} classes, expected {C}")
    target = _metrics_target(target, (B, H, W))
    _cuda(target)
    check(lib.b200seg_seg_metrics(ptr(logits), _dt(logits), _cabi.NHWC if nhwc else _cabi.NCHW, ldc, ptr(target),
                                  _TGT[target.dtype], int(ignore_index), ptr(confusion), ptr(counts), ptr(loss_sum),
                                  B, C, H, W, _stream()), "seg_metrics")


def nhwc_to_nchw(x, C: int, out_dtype, out=None):
    _cuda(x)
    B, H, W, ldc = x.shape
    if out is None:
        out = torch.empty((B, C, H, W), device=x.device, dtype=out_dtype)
    check(lib.b200seg_nhwc_to_nchw(ptr(x), _dt(x), ldc, ptr(out), _dt(out), B, H, W, C, _stream()), "nhwc_to_nchw")
    return out


def nhwc_argmax(x, C: int, out=None):
    """uint8 [B,H,W] = argmax over the first C channels of NHWC x (first maximum wins, like torch.max)."""
    _cuda(x)
    B, H, W, ldc = x.shape
    if out is None:
        out = torch.empty((B, H, W), device=x.device, dtype=torch.uint8)
    check(lib.b200seg_nhwc_argmax(ptr(x), _dt(x), ldc, ptr(out), B * H * W, C, _stream()), "nhwc_argmax")
    return out


def maxpool2x2(x, out=None):
    _cuda(x)
    B, H, W, Cc = x.shape
    if out is None:
        out = torch.empty((B, H // 2, W // 2, Cc), device=x.device, dtype=x.dtype)
    check(lib.b200seg_maxpool2x2(ptr(x), ptr(out), _dt(x), B, H, W, Cc, _stream()), "maxpool2x2")
    return out


IGNORE_INDEX = -100      # nn.CrossEntropyLoss default


def softmax_ce(logits, target, want_grad: bool = True, grad_scale: Optional[float] = None):
    """Fused mean cross-entropy over NCHW f32 logits and int64 targets (nn.CrossEntropyLoss defaults: 'mean' over the
    targets that are not ignore_index=-100).  Returns (loss scalar tensor, dlogits or None); dlogits already carries
    the 1/n_valid factor.  A label outside [0,C) that is not ignore_index makes the loss NaN (torch asserts on the
    device; neither may silently train on a broken label map).  ``grad_scale`` (tests): plain factor, no counting."""
    _cuda(logits, target)
    if logits.dtype != torch.float32 or target.dtype != torch.int64:
        raise TypeError("softmax_ce expects f32 logits and int64 targets")
    B, Cc, H, W = logits.shape
    n = B * H * W
    acc = torch.zeros(3, device=logits.device, dtype=torch.float32)      # [loss sum, valid targets, bad labels]
    dl = torch.empty_like(logits) if want_grad else None
    if grad_scale is None:
        check(lib.b200seg_ce_count(ptr(target), ptr(acc[1:]), n, Cc, IGNORE_INDEX, _stream()), "ce_count")
        check(lib.b200seg_softmax_ce(ptr(logits), ptr(target), ptr(acc), ptr(dl), 1.0, ptr(acc[1:]), B, Cc, H, W, _stream()),
              "softmax_ce")
        loss = acc[0] / acc[1]                                            # 0/0 = NaN for an all-ignored batch, as torch
        return torch.where(acc[2] > 0, torch.full_like(loss, float("nan")), loss), dl
    check(lib.b200seg_softmax_ce(ptr(logits), ptr(target), ptr(acc), ptr(dl), grad_scale, None, B, Cc, H, W, _stream()),
          "softmax_ce")
    return acc[0] / n, dl


_TGT = {torch.int64: _cabi.I64, torch.uint8: _cabi.U8}


def _ce_ex_args(logits, target, weight):
    _cuda(logits, target, weight)
    if logits.dtype != torch.float32 or logits.dim() != 4:
        raise TypeError("softmax_ce_ex expects f32 NCHW logits")
    if target.dtype not in _TGT:
        raise TypeError(f"softmax_ce_ex: targets must be int64 or uint8, got {target.dtype}")
    B, Cc, H, W = logits.shape
    if tuple(target.shape) != (B, H, W):
        raise ValueError(f"softmax_ce_ex: target shape {tuple(target.shape)} does not match logits {tuple(logits.shape)}")
    if weight is not None:
        if weight.dtype != torch.float32 or weight.dim() != 1 or weight.numel() != Cc:
            raise ValueError(f"softmax_ce_ex: weight must be f32 [C={Cc}], got {weight.dtype} {tuple(weight.shape)}")
        if weight.device != logits.device:
            raise RuntimeError(f"softmax_ce_ex: weight on {weight.device}, logits on {logits.device}")
    return B, Cc, H, W, _TGT[target.dtype]


def softmax_ce_ex(logits, target, weight=None, ignore_index: int = IGNORE_INDEX, label_smoothing: float = 0.0,
                  reduction: str = "mean", want_grad: bool = True):
    """nn.CrossEntropyLoss(weight, ignore_index, reduction, label_smoothing) over NCHW f32 logits and int64 or uint8
    targets (csrc/softmax_ce_ex.cu).  Returns (loss, dlogits or None).  'mean' / 'sum': a scalar, and dlogits of that
    scalar from the same pass ('mean' divides by the weight sum of the counted targets, from b200seg_ce_count_ex).
    'none': the f32 [B,H,W] loss map and no dlogits (softmax_ce_ex_backward gives them for an incoming gradient).  A
    label outside [0,C) that is not ignore_index makes the loss NaN (per pixel for 'none')."""
    B, Cc, H, W, tdt = _ce_ex_args(logits, target, weight)
    if reduction == "none":
        out = torch.empty((B, H, W), device=logits.device, dtype=torch.float32)
        check(lib.b200seg_softmax_ce_ex(ptr(logits), ptr(target), tdt, ignore_index, ptr(weight), label_smoothing, None,
                                        ptr(out), None, None, B, Cc, H, W, _stream()), "softmax_ce_ex")
        return out, None
    if reduction not in ("mean", "sum"):
        raise ValueError(f"{reduction} is not a valid value for reduction")
    acc = torch.zeros(3, device=logits.device, dtype=torch.float64)      # [loss sum, sum of w_t counted, bad labels]
    dl = torch.empty_like(logits) if want_grad else None
    if reduction == "mean":
        check(lib.b200seg_ce_count_ex(ptr(target), tdt, ignore_index, ptr(weight), ptr(acc[1:]), B * H * W, Cc, _stream()),
              "ce_count_ex")
    check(lib.b200seg_softmax_ce_ex(ptr(logits), ptr(target), tdt, ignore_index, ptr(weight), label_smoothing, ptr(acc), None,
                                    ptr(dl), ptr(acc[1:]) if reduction == "mean" else None, B, Cc, H, W, _stream()),
          "softmax_ce_ex")
    loss = acc[0] / acc[1] if reduction == "mean" else acc[0]           # 0/0 = NaN for an all-ignored batch, as torch
    return loss.float(), dl


def softmax_ce_ex_backward(logits, target, gout, weight=None, ignore_index: int = IGNORE_INDEX, label_smoothing: float = 0.0):
    """d(sum(loss_map * gout)) / d(logits) of softmax_ce_ex(..., reduction='none'), one pass over the logits."""
    B, Cc, H, W, tdt = _ce_ex_args(logits, target, weight)
    _cuda(gout)
    if gout.dtype != torch.float32 or tuple(gout.shape) != (B, H, W):
        raise ValueError(f"softmax_ce_ex_backward: gout must be f32 {(B, H, W)}")
    dl = torch.empty_like(logits)
    check(lib.b200seg_softmax_ce_ex_bwd(ptr(logits), ptr(target), tdt, ignore_index, ptr(weight), label_smoothing, ptr(gout),
                                        ptr(dl), B, Cc, H, W, _stream()), "softmax_ce_ex_bwd")
    return dl


def scale_unless_one(x, s):
    """x *= s (device scalar) in place; nothing is read or written when s == 1."""
    _cuda(x, s)
    if x.dtype != torch.float32 or s.dtype != torch.float32 or not x.is_contiguous():
        raise TypeError("scale_unless_one: contiguous f32 tensors")
    check(lib.b200seg_scale_unless_one(ptr(x), x.numel(), ptr(s), _stream()), "scale_unless_one")
    return x


# ------------------------------------------------------------------------------------------------
# training-path wrappers (train.py:35-39).  Activations are NHWC [B,H,W,C]; P = B*H*W.
# ------------------------------------------------------------------------------------------------
# copies of every per-channel reduction output (see include/b200seg.h): CTA i adds into copy i % NSLOT
NSLOT = 16


class _ZeroPool:
    """Zero-initialised f64 accumulators carved out of few large memsets (one fill kernel per 8 MB instead of one per
    reduction: ~200 fewer launches per training step).  A slice is handed out once; ``reset()`` at the start of a
    pass drops the current chunk so that a CUDA-graph capture never inherits memory zeroed outside the graph."""

    def __init__(self, dtype=torch.float64, chunk=1 << 20):
        self.buf, self.off, self.dtype, self.CHUNK = None, 0, dtype, chunk

    def reset(self):
        self.buf, self.off = None, 0

    def take(self, shape, device) -> torch.Tensor:
        n = 1
        for d in shape:
            n *= int(d)
        if self.buf is None or self.buf.device != device or self.off + n > self.buf.numel():
            self.buf = torch.zeros(max(n, self.CHUNK), device=device, dtype=self.dtype)
            self.off = 0
        t = self.buf[self.off:self.off + n].view(*shape)
        self.off += (n + 3) // 4 * 4           # keep 16-byte alignment
        return t


zero_pool = _ZeroPool()
zero_pool32 = _ZeroPool(torch.float32, 4 << 20)      # weight-gradient accumulators (26 MB per step)


def _P(t):
    return t.shape[0] * t.shape[1] * t.shape[2]


BN_CLUSTER = True        # small / mid-size bf16 layers: one cluster-synchronised launch per direction (csrc/bn_cluster.cu)


# large-layer BatchNorm: per-channel constants derived inside the apply kernels (no bn_finalize / f64->f32 launches)
BN_FUSED_CONST = os.environ.get("B200SEG_BN_FUSED_CONST", "1") != "0"


def bn_train_forward(z, gamma, beta, running_mean, running_var, eps: float, momentum: float, act: int, res=None):
    """Train-mode BatchNorm over NHWC z (+act, +residual).  Updates the running stats in place.
    Returns (a, saved) where saved = (mean, invstd, scale, shift) for the backward pass.
    (Finishing the statistics in the reduction kernel itself -- "last block done" -- was measured SLOWER than the separate
    one-block finalize launch: the ticket fence and the finalize code's registers cost the streaming loop more than the
    5 us launch gap they remove; bn_stats 0.61 + finalize 0.35 ms vs 1.05-1.20 ms fused, per training step.)"""
    _cuda(z, gamma, beta, running_mean, running_var, res)
    C, P = z.shape[-1], _P(z)
    if BN_CLUSTER and lib.b200seg_bn_cluster_supported(_dt(z), P, C):
        sv = torch.empty(4, C, device=z.device, dtype=torch.float32)
        a = torch.empty_like(z)
        check(lib.b200seg_bn_cluster_fwd(ptr(z), P, C, ptr(gamma), ptr(beta), eps, momentum, ptr(running_mean), ptr(running_var),
                                         ptr(sv), ptr(res), ptr(a), act, _stream()), "bn_cluster_fwd")
        return a, sv
    st = zero_pool.take((NSLOT, 2, C), z.device)                              # slot-major: [slot][sum | sumsq][C]
    check(lib.b200seg_bn_stats(ptr(z), _dt(z), P, C, ptr(st[0, 0]), ptr(st[0, 1]), NSLOT, 2 * C, _stream()), "bn_stats")
    sv = torch.empty(4, C, device=z.device, dtype=torch.float32)
    if BN_FUSED_CONST:        # finalize inside the apply launch (every block repeats the per-channel arithmetic)
        a = torch.empty_like(z)
        check(lib.b200seg_bn_finalize_apply(ptr(z), ptr(st), NSLOT, ptr(gamma), ptr(beta), eps, momentum, ptr(running_mean),
                                            ptr(running_var), ptr(sv), ptr(res), ptr(a), _dt(z), P, C, act, _stream()),
              "bn_finalize_apply")
        return a, sv
    check(lib.b200seg_bn_finalize(ptr(z), _dt(z), ptr(st[0, 0]), ptr(st[0, 1]), NSLOT, 2 * C, P, ptr(gamma), ptr(beta), eps, momentum, ptr(running_mean),
                                  ptr(running_var), ptr(sv[0]), ptr(sv[1]), ptr(sv[2]), ptr(sv[3]), C, _stream()),
          "bn_finalize")
    a = torch.empty_like(z)
    check(lib.b200seg_bn_apply(ptr(z), ptr(sv[2]), ptr(sv[3]), ptr(res), ptr(a), _dt(z), P, C, act, _stream()), "bn_apply")
    return a, sv


def bn_train_backward(da, z, sv, act: int, red=None):
    """Returns (dz, dgamma f32[C], dbeta f32[C]).  ``red``: zeroed f64 staging [NSLOT, 2, C] that receives the slot sums
    (row 0 = d beta, row 1 = d gamma; the gradient-finalize kernel reads them from there)."""
    _cuda(da, z, sv)
    C, P = z.shape[-1], _P(z)
    own_red = red is None
    if red is None:
        red = zero_pool.take((NSLOT, 2, C), z.device)
    if BN_CLUSTER and lib.b200seg_bn_cluster_bwd_supported(_dt(z), P, C):
        dz = torch.empty_like(z)
        check(lib.b200seg_bn_cluster_bwd(ptr(da), ptr(z), ptr(sv), P, C, act, ptr(red), ptr(dz), _stream()), "bn_cluster_bwd")
        if not own_red:               # the training step reads the sums from the staging block (gradient finalize)
            return dz, None, None
        g32 = red[0].float()
        return dz, g32[1], g32[0]
    check(lib.b200seg_bn_bwd_reduce(ptr(da), ptr(z), ptr(sv[2]), ptr(sv[3]), ptr(sv[0]), ptr(sv[1]), _dt(z), P, C, act,
                                    ptr(red[0, 0]), ptr(red[0, 1]), NSLOT, 2 * C, _stream()), "bn_bwd_reduce")
    if BN_FUSED_CONST and not own_red:      # the training step: the apply pass sums the f64 slots itself
        dz = torch.empty_like(z)
        check(lib.b200seg_bn_bwd_apply_slots(ptr(da), ptr(z), ptr(sv), ptr(red), NSLOT, ptr(dz), _dt(z), P, C, act, _stream()),
              "bn_bwd_apply_slots")
        return dz, None, None
    g32 = torch.empty(2, C, device=z.device, dtype=torch.float32)
    check(lib.b200seg_f64_to_f32(ptr(red), ptr(g32), 2 * C, NSLOT, 2 * C, 1.0, _stream()), "f64_to_f32")
    dz = torch.empty_like(z)
    check(lib.b200seg_bn_bwd_apply(ptr(da), ptr(z), ptr(sv[2]), ptr(sv[3]), ptr(sv[0]), ptr(sv[1]), ptr(g32[0]), ptr(g32[1]),
                                   ptr(dz), _dt(z), P, C, act, _stream()), "bn_bwd_apply")
    return dz, g32[1], g32[0]


def act_bwd(da, a_out, act: int):
    _cuda(da, a_out)
    dz = torch.empty_like(da)
    check(lib.b200seg_act_bwd(ptr(da), ptr(a_out), ptr(dz), _dt(da), da.numel(), act, _stream()), "act_bwd")
    return dz


def colsum(x, acc=None):
    """f32 [C] = sum over pixels of NHWC x.  With ``acc`` (zeroed f64 staging [NSLOT, C]) only the slot sums are
    produced (returns None)."""
    _cuda(x)
    C = x.shape[-1]
    if acc is not None:
        check(lib.b200seg_colsum(ptr(x), _dt(x), _P(x), C, ptr(acc), NSLOT, C, _stream()), "colsum")
        return None
    acc = zero_pool.take((NSLOT, C), x.device)
    check(lib.b200seg_colsum(ptr(x), _dt(x), _P(x), C, ptr(acc), NSLOT, C, _stream()), "colsum")
    out = torch.empty(C, device=x.device, dtype=torch.float32)
    check(lib.b200seg_f64_to_f32(ptr(acc), ptr(out), C, NSLOT, C, 1.0, _stream()), "f64_to_f32")
    return out


def conv_wgrad(x, dz, taps: int, dw=None):
    """f32 [Cout, taps*Cin] = sum_p dz[p] (outer) im2col(x)[p]  (``dw``: zeroed accumulator to add into)."""
    _cuda(x, dz)
    B, H, W, Cin = x.shape
    Cout = dz.shape[-1]
    if dw is None:
        dw = zero_pool32.take((Cout, taps * Cin), x.device)
    check(lib.b200seg_conv_wgrad(ptr(x), ptr(dz), ptr(dw), _dt(x), B, H, W, Cin, Cout, taps, _stream()), "conv_wgrad")
    return dw


def conv_wgrad_tc(x, dz, taps: int, dw=None):
    """Tensor-core weight gradient: bf16 NHWC x / dz -> f32 [Cout, taps*Cin]  (``dw``: zeroed accumulator)."""
    _cuda(x, dz)
    if x.dtype != torch.bfloat16 or dz.dtype != torch.bfloat16:
        raise TypeError("conv_wgrad_tc is bf16-only")
    B, H, W, Cin = x.shape
    Cout = dz.shape[-1]
    if dw is None:
        dw = zero_pool32.take((Cout, taps * Cin), x.device)
    check(lib.b200seg_conv_wgrad_tc(ptr(x), ptr(dz), ptr(dw), B, H, W, Cin, Cout, taps, _stream()), "conv_wgrad_tc")
    return dw


def dw_dgrad(dz, w9c, in_shape, stride: int, acc=None):
    _cuda(dz, w9c, acc)
    B, H, W, Cc = in_shape
    dx = torch.empty(in_shape, device=dz.device, dtype=dz.dtype)
    check(lib.b200seg_dw_dgrad(ptr(dz), ptr(w9c), ptr(acc), ptr(dx), _dt(dz), B, H, W, Cc, stride, _stream()), "dw_dgrad")
    return dx


def dw_wgrad(x, dz, stride: int, acc=None):
    """f32 [9, C].  With ``acc`` (zeroed f64 staging [NSLOT, 9, C]) only the slot sums are produced (returns None)."""
    _cuda(x, dz)
    B, H, W, Cc = x.shape
    if acc is not None:
        check(lib.b200seg_dw_wgrad(ptr(x), ptr(dz), ptr(acc), NSLOT, _dt(x), B, H, W, Cc, stride, _stream()), "dw_wgrad")
        return None
    acc = zero_pool.take((NSLOT, 9, Cc), x.device)
    check(lib.b200seg_dw_wgrad(ptr(x), ptr(dz), ptr(acc), NSLOT, _dt(x), B, H, W, Cc, stride, _stream()), "dw_wgrad")
    out = torch.empty(9, Cc, device=x.device, dtype=torch.float32)
    check(lib.b200seg_f64_to_f32(ptr(acc), ptr(out), 9 * Cc, NSLOT, 9 * Cc, 1.0, _stream()), "f64_to_f32")
    return out


def smallcin_wgrad(x_nchw, dz, stride: int, dw=None):
    """f32 [3,3,Cin,Cout]  (``dw``: zeroed accumulator)."""
    _cuda(x_nchw, dz)
    B, Cin, H, W = x_nchw.shape
    Cout = dz.shape[-1]
    if dw is None:
        dw = zero_pool32.take((3, 3, Cin, Cout), dz.device)
    check(lib.b200seg_smallcin_wgrad(ptr(x_nchw), _dt(x_nchw), ptr(dz), _dt(dz), ptr(dw), B, Cin, H, W, Cout, stride,
                                     _stream()), "smallcin_wgrad")
    return dw


def upcat_bwd(dcat, Cs: int, acc_skip=None):
    """Returns (dskip [B,2h,2w,Cs] (+acc_skip), dx [B,h,w,Cu])."""
    _cuda(dcat, acc_skip)
    B, H2, W2, Cc = dcat.shape
    h, w, Cu = H2 // 2, W2 // 2, Cc - Cs
    dskip = torch.empty(B, H2, W2, Cs, device=dcat.device, dtype=dcat.dtype)
    dx = torch.empty(B, h, w, Cu, device=dcat.device, dtype=dcat.dtype)
    check(lib.b200seg_upcat_bwd(ptr(dcat), ptr(acc_skip), ptr(dskip), ptr(dx), _dt(dcat), B, h, w, Cs, Cu, _stream()),
          "upcat_bwd")
    return dskip, dx


def final_bwd(dout_nchw, sdt, ldc: int = 16, out=None):
    """dout NCHW f32 [B,C,2h,2w] -> NHWC [B,h,w,ldc] of dtype sdt (``out``: existing result buffer)."""
    _cuda(dout_nchw)
    if dout_nchw.dtype != torch.float32:
        raise TypeError("final_bwd expects f32 upstream gradients")
    B, Cc, H2, W2 = dout_nchw.shape
    dl = out if out is not None else torch.empty(B, H2 // 2, W2 // 2, ldc, device=dout_nchw.device, dtype=sdt)
    if tuple(dl.shape) != (B, H2 // 2, W2 // 2, ldc) or dl.dtype != sdt or not dl.is_contiguous():
        raise ValueError("final_bwd: bad output buffer")
    if ldc != 16:
        check(lib.b200seg_final_bwd_generic(ptr(dout_nchw), ptr(dl), _dt(dl), B, H2 // 2, W2 // 2, Cc, ldc, _stream()),
              "final_bwd_generic")
        return dl
    check(lib.b200seg_final_bwd(ptr(dout_nchw), ptr(dl), _dt(dl), B, H2 // 2, W2 // 2, Cc, _stream()), "final_bwd")
    return dl


def nchw_to_nhwc_pad(x_nchw, ldc: int, sdt, out=None):
    _cuda(x_nchw)
    B, Cc, H, W = x_nchw.shape
    y = out if out is not None else torch.empty(B, H, W, ldc, device=x_nchw.device, dtype=sdt)
    if tuple(y.shape) != (B, H, W, ldc) or y.dtype != sdt or not y.is_contiguous():
        raise ValueError("nchw_to_nhwc_pad: bad output buffer")
    check(lib.b200seg_nchw_to_nhwc_pad(ptr(x_nchw), ptr(y), _dt(y), B, Cc, H, W, ldc, _stream()), "nchw_to_nhwc_pad")
    return y


def maxpool_bwd(x, dy, acc=None):
    _cuda(x, dy, acc)
    B, H, W, Cc = x.shape
    dx = torch.empty_like(x)
    check(lib.b200seg_maxpool_bwd(ptr(x), ptr(dy), ptr(acc), ptr(dx), _dt(x), B, H, W, Cc, _stream()), "maxpool_bwd")
    return dx
