"""detect_objects / overlay argument checking without a GPU: the C entry points reject bad arguments before any CUDA call,
and the Python functions validate dtype, device and classes before touching the device."""
import ctypes

import pytest
import torch

import b200seg
from b200seg import _cabi

lib = _cabi.lib
FAKE = 1 << 20             # a non-null device address; never dereferenced because the checks fail first


def _detect(B=1, Hm=8, Wm=8, H=8, W=8, classes=(1,), K=None, close=5, max_objects=4, mask=FAKE, ws=FAKE, count=FAKE):
    arr = (ctypes.c_int * max(1, len(classes)))(*classes) if classes is not None else None
    K = len(classes) if K is None else K
    return lib.b200seg_detect_objects(mask, B, Hm, Wm, H, W, arr, K, close, 0, max_objects, ws, 1 << 40, count, FAKE, FAKE,
                                      None, None)


def _err():
    return lib.b200seg_last_error().decode()


@pytest.mark.parametrize("K", [0, 17])
def test_class_count_outside_1_to_16(K):
    cls = tuple(range(max(K, 1)))
    assert _detect(classes=cls, K=K) < 0
    assert "classes" in _err()


@pytest.mark.parametrize("close", [0, 2, 4, 16, 17, -1])
def test_even_or_oversized_close(close):
    assert _detect(close=close) < 0
    assert "close" in _err()


def test_null_pointers_and_sizes():
    assert _detect(mask=None) < 0 and "null" in _err()
    assert _detect(ws=None) < 0 and "null" in _err()
    assert _detect(count=None) < 0 and "null" in _err()
    assert _detect(classes=None, K=1) < 0 and "null" in _err()
    for kw in (dict(B=0), dict(H=0), dict(W=-3), dict(Hm=0), dict(Wm=-1)):
        assert _detect(**kw) < 0, kw
        assert "non-positive" in _err(), kw
    assert _detect(max_objects=0) < 0 and "max_objects" in _err()
    assert _detect(classes=(1, 2, 1)) < 0 and "twice" in _err()
    assert _detect(classes=(256,)) < 0 and "[0, 255]" in _err()
    assert _detect(classes=(-1,)) < 0


def test_workspace_size_and_its_errors():
    n = ctypes.c_longlong(0)
    assert lib.b200seg_detect_workspace_bytes(64, 9, 540, 960, ctypes.byref(n)) == 0
    nb = 270 * 480
    assert n.value >= 64 * 540 * 960 * 2 + 64 * 9 * nb * (4 + 4 + 40)    # bits, parents, ids, statistics slots
    assert lib.b200seg_detect_workspace_bytes(1, 17, 8, 8, ctypes.byref(n)) < 0
    assert lib.b200seg_detect_workspace_bytes(1, 1, 0, 8, ctypes.byref(n)) < 0
    assert lib.b200seg_detect_workspace_bytes(1, 1, 8, 8, None) < 0
    # a workspace smaller than the size asked for is refused
    cls = (ctypes.c_int * 1)(1)
    rc = lib.b200seg_detect_objects(FAKE, 1, 8, 8, 8, 8, cls, 1, 5, 0, 4, FAKE, 16, FAKE, FAKE, FAKE, None, None)
    assert rc < 0 and "workspace" in _err()


def test_overlay_argument_errors():
    f = ctypes.c_float
    args = lambda **kw: [kw.get("frames", FAKE), kw.get("mask", FAKE), kw.get("B", 1), 4, 4, kw.get("H", 8), 8,
                         kw.get("pal", FAKE), kw.get("npal", 3), f(0.5), f(0.5), f(0.0), kw.get("out", FAKE), None]
    assert lib.b200seg_overlay(*args(frames=None)) < 0 and "null" in _err()
    assert lib.b200seg_overlay(*args(out=None)) < 0
    assert lib.b200seg_overlay(*args(pal=None)) < 0
    assert lib.b200seg_overlay(*args(B=0)) < 0 and "non-positive" in _err()
    assert lib.b200seg_overlay(*args(H=-1)) < 0
    assert lib.b200seg_overlay(*args(npal=257)) < 0 and "palette" in _err()


def test_python_side_errors_before_the_device():
    m = torch.zeros(1, 8, 8, dtype=torch.uint8)
    with pytest.raises(ValueError, match="uint8"):
        b200seg.detect_objects(m.float(), [1])                             # dtype
    with pytest.raises(ValueError, match="uint8"):
        b200seg.detect_objects(m[0], [1])                                  # not [B,H,W]
    with pytest.raises(RuntimeError, match="CUDA"):
        b200seg.detect_objects(m, [1])                                     # CPU tensor: no fallback
    with pytest.raises(ValueError, match="duplicate"):
        b200seg.detect_objects(m, [1, 2, 1])
    with pytest.raises(ValueError):
        b200seg.detect_objects(m, list(range(17)))
    with pytest.raises(ValueError):
        b200seg.detect_objects(m, [])
    with pytest.raises(ValueError):
        b200seg.detect_objects(m, [300])
    with pytest.raises(ValueError, match="close"):
        b200seg.detect_objects(m, [1], close=6)
    with pytest.raises(ValueError):
        b200seg.detect_objects(m, [1], max_objects=0)
    with pytest.raises(ValueError):
        b200seg.detect_objects(m, [1], size=(0, 8))
    frames = torch.zeros(1, 8, 8, 3, dtype=torch.uint8)
    with pytest.raises(ValueError):
        b200seg.overlay(frames.float(), m, [[0, 0, 0]], 0.5, 0.5)
    with pytest.raises(ValueError):
        b200seg.overlay(frames, m.float(), [[0, 0, 0]], 0.5, 0.5)
    with pytest.raises(ValueError):
        b200seg.overlay(frames, torch.zeros(2, 8, 8, dtype=torch.uint8), [[0, 0, 0]], 0.5, 0.5)
    with pytest.raises(RuntimeError, match="CUDA"):
        b200seg.overlay(frames, m, [[0, 0, 0]], 0.5, 0.5)
