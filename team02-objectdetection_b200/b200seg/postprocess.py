"""Object boxes and the colour overlay on the GPU: the post-processing of the inference script (inference.py:48-146,
``overlay_predictions``), batched.

    mask = model.predict_mask(x)                                          # uint8 [B,Hm,Wm]
    det = b200seg.detect_objects(mask, classes=range(1, 10), size=(960, 540), close=5, min_area=100)
    for frame_rows in det.to_list():                                      # one device-to-host copy
        for cls, label, left, top, width, height, area, cx, cy in frame_rows:
            ...
    vis = b200seg.overlay(frames, mask, palette, 0.7, 0.3)               # uint8 [B,H,W,3] BGR

Each step equals the cv2 call the reference makes, value for value: ``cv2.resize(mask, size, INTER_NEAREST)``, per class
``cv2.morphologyEx(resized == cls, MORPH_CLOSE, np.ones((close, close)))`` and
``cv2.connectedComponentsWithStats(closed, connectivity=8)`` (labels numbered as cv2 numbers them), and
``cv2.addWeighted(frame, alpha, palette[resized], beta, gamma)``.  Both functions enqueue kernels on the current stream of
the tensor's device, never synchronise with the host and can be captured in a CUDA graph.
"""
from __future__ import annotations

import ctypes

import torch

from ._cabi import check, lib, ptr

MAX_CLASSES = 16          # one bit per selected class in a uint16 per pixel
MAX_CLOSE = 15


class Detections:
    """Result of :func:`detect_objects`, on the device.

    ``count``    int32 [B]: components with ``area >= min_area`` per frame (may exceed ``max_objects``)
    ``stats``    int32 [B, max_objects, 7]: class, cv2 label, left, top, width, height, area; rows past the count are 0
    ``centroid`` float64 [B, max_objects, 2]: x, y (the coordinate sums over the area, as cv2 computes them)
    ``labels``   int32 [B, K, H, W]: the cv2 label image of every selected class, or None
    Within a frame the rows are ordered by the class's position in ``classes``, then by cv2 label."""

    def __init__(self, buf: torch.Tensor, B: int, M: int, classes, labels):
        self._buf = buf                     # [centroid f64 | stats i32 | count i32]: one copy brings everything to the host
        self.max_objects = M
        self.classes = tuple(classes)
        self.centroid = buf[:B * M * 16].view(torch.float64).view(B, M, 2)
        self.stats = buf[B * M * 16:B * M * 44].view(torch.int32).view(B, M, 7)
        self.count = buf[B * M * 44:B * M * 44 + 4 * B].view(torch.int32)
        self.labels = labels

    def to_list(self):
        """Host rows, one list per frame of ``(class, label, left, top, width, height, area, cx, cy)`` tuples (at most
        ``max_objects``).  This is the one device-to-host copy and the one synchronisation of the flow."""
        B, M = self.count.shape[0], self.max_objects
        host = self._buf.cpu()
        cen = host[:B * M * 16].view(torch.float64).view(B, M, 2).tolist()
        st = host[B * M * 16:B * M * 44].view(torch.int32).view(B, M, 7).tolist()
        cnt = host[B * M * 44:B * M * 44 + 4 * B].view(torch.int32).tolist()
        return [[tuple(st[b][r]) + tuple(cen[b][r]) for r in range(min(cnt[b], M))] for b in range(B)]

    def __repr__(self):
        return f"Detections(frames={self.count.shape[0]}, max_objects={self.max_objects}, classes={self.classes})"


def _check_mask(mask, what):
    if not torch.is_tensor(mask) or mask.dtype != torch.uint8 or mask.dim() != 3:
        got = f"{tuple(mask.shape)} {mask.dtype}" if torch.is_tensor(mask) else type(mask).__name__
        raise ValueError(f"{what}: expected a uint8 class mask [B,H,W] (what predict_mask returns), got {got}")
    if min(mask.shape) < 1:
        raise ValueError(f"{what}: empty mask {tuple(mask.shape)}")


def _check_cuda(t, what):
    if not t.is_cuda:
        raise RuntimeError(f"{what} runs on CUDA tensors only (sm_100a); got a CPU tensor. There is deliberately no CPU fallback.")


def _frame_size(mask, size):
    if size is None:
        return int(mask.shape[1]), int(mask.shape[2])
    W, H = int(size[0]), int(size[1])                  # cv2 order: (width, height)
    if W < 1 or H < 1:
        raise ValueError(f"size must be positive (width, height), got {tuple(size)}")
    return H, W


def detect_objects(mask: torch.Tensor, classes, size=None, close: int = 5, min_area: int = 0, max_objects: int = 256,
                   labels: bool = False) -> Detections:
    """Connected components with statistics of the closed class planes of ``mask`` (uint8 [B,Hm,Wm] CUDA tensor).

    ``classes``: 1..16 distinct class ids in [0, 255]; ``size``: the frame size (width, height) the mask is resized to with
    nearest-neighbour sampling (default: the mask's own size); ``close``: the side of the square closing element (odd,
    1..15; 1 = no closing); ``min_area``: the smallest component area reported; ``max_objects``: the rows kept per frame;
    ``labels``: also return the label image of every plane.  See :class:`Detections`."""
    _check_mask(mask, "detect_objects")
    try:
        classes = [int(c) for c in classes]
    except TypeError:
        raise ValueError(f"classes must be a sequence of ints, got {classes!r}") from None
    if not 1 <= len(classes) <= MAX_CLASSES:
        raise ValueError(f"detect_objects takes 1..{MAX_CLASSES} classes, got {len(classes)}")
    if len(set(classes)) != len(classes):
        raise ValueError(f"duplicate class ids in {classes}")
    if any(c < 0 or c > 255 for c in classes):
        raise ValueError(f"class ids must be in [0, 255], got {classes}")
    close = int(close)
    if close < 1 or close > MAX_CLOSE or close % 2 == 0:
        raise ValueError(f"close must be odd and in 1..{MAX_CLOSE}, got {close}")
    max_objects = int(max_objects)
    if max_objects < 1:
        raise ValueError(f"max_objects must be >= 1, got {max_objects}")
    H, W = _frame_size(mask, size)
    _check_cuda(mask, "detect_objects")
    mask = mask.contiguous()
    B, Hm, Wm = mask.shape
    K = len(classes)
    nbytes = ctypes.c_longlong(0)
    check(lib.b200seg_detect_workspace_bytes(B, K, H, W, ctypes.byref(nbytes)), "detect_workspace_bytes")
    dev = mask.device
    ws = torch.empty(nbytes.value + 256, dtype=torch.uint8, device=dev)
    w0 = (-ws.data_ptr()) % 256                          # 256-byte aligned start
    buf = torch.empty(B * max_objects * 44 + 4 * B, dtype=torch.uint8, device=dev)
    lab = torch.empty((B, K, H, W), dtype=torch.int32, device=dev) if labels else None
    det = Detections(buf, B, max_objects, classes, lab)
    cls = (ctypes.c_int * K)(*classes)
    with torch.cuda.device(dev):                         # launch on the mask's device, whatever the current one is
        check(lib.b200seg_detect_objects(ptr(mask), B, Hm, Wm, H, W, cls, K, close, int(min_area), max_objects,
                                         ws.data_ptr() + w0, nbytes.value, ptr(det.count), ptr(det.stats), ptr(det.centroid),
                                         ptr(lab), torch.cuda.current_stream().cuda_stream), "detect_objects")
    return det


def overlay(frames: torch.Tensor, mask: torch.Tensor, palette, alpha: float, beta: float, gamma: float = 0.0,
            out: torch.Tensor = None) -> torch.Tensor:
    """``cv2.addWeighted(frame, alpha, palette[cv2.resize(mask, INTER_NEAREST)], beta, gamma)`` for every frame.

    ``frames``: uint8 BGR [B,H,W,3] CUDA tensor; ``mask``: uint8 [B,Hm,Wm] on the same device; ``palette``: up to 256 BGR
    colours, uint8 [P,3] (a CUDA tensor keeps the call capturable; anything else is copied to the device first).  Mask
    values with no palette row blend with black.  Returns ``out`` (uint8 [B,H,W,3], allocated if None)."""
    if not torch.is_tensor(frames) or frames.dtype != torch.uint8 or frames.dim() != 4 or frames.shape[-1] != 3:
        got = f"{tuple(frames.shape)} {frames.dtype}" if torch.is_tensor(frames) else type(frames).__name__
        raise ValueError(f"overlay: expected uint8 BGR frames [B,H,W,3], got {got}")
    _check_mask(mask, "overlay")
    if mask.shape[0] != frames.shape[0]:
        raise ValueError(f"overlay: {frames.shape[0]} frames but {mask.shape[0]} masks")
    _check_cuda(frames, "overlay")
    _check_cuda(mask, "overlay")
    if mask.device != frames.device:
        raise ValueError(f"overlay: frames on {frames.device}, mask on {mask.device}")
    pal = palette if torch.is_tensor(palette) else torch.as_tensor(palette, dtype=torch.uint8)
    if pal.dtype != torch.uint8 or pal.dim() != 2 or pal.shape[1] != 3 or pal.shape[0] > 256:
        raise ValueError(f"overlay: palette must be uint8 [P,3] with P <= 256, got {tuple(pal.shape)} {pal.dtype}")
    pal = pal.to(frames.device).contiguous()
    frames, mask = frames.contiguous(), mask.contiguous()
    B, H, W, _ = frames.shape
    if out is None:
        out = torch.empty_like(frames)
    elif out.dtype != torch.uint8 or tuple(out.shape) != tuple(frames.shape) or not out.is_contiguous() or out.device != frames.device:
        raise ValueError(f"overlay: out must be a contiguous uint8 {tuple(frames.shape)} tensor on {frames.device}")
    f = ctypes.c_float
    with torch.cuda.device(frames.device):
        check(lib.b200seg_overlay(ptr(frames), ptr(mask), B, mask.shape[1], mask.shape[2], H, W, ptr(pal), pal.shape[0],
                                  f(alpha), f(beta), f(gamma), ptr(out), torch.cuda.current_stream().cuda_stream), "overlay")
    return out
