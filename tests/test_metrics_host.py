"""SegmentationMetrics host logic on the CPU: compute() on hand-built states, the one-collective all_reduce over gloo
(world size 2), and the argument checks of the two metrics entry points of the C ABI (before any CUDA call)."""
import math
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import b200seg
from b200seg import _cabi


def _metrics(cm, valid, invalid, loss_sum):
    C = len(cm)
    m = b200seg.SegmentationMetrics(C, device="cpu")
    m.confusion.copy_(torch.tensor(cm, dtype=torch.int64))
    m.counts.copy_(torch.tensor([valid, invalid], dtype=torch.int64))
    m.loss_sum.fill_(loss_sum)
    return m


def test_compute_iou_accuracy_and_loss():
    # class 2 is absent from targets and predictions: NaN IoU, left out of the mean
    r = _metrics([[5, 1, 0], [2, 4, 0], [0, 0, 0]], 12, 0, 6.0).compute()
    assert r["valid"] == 12 and r["invalid"] == 0
    assert math.isclose(r["loss"], 0.5)
    assert math.isclose(r["pixel_accuracy"], 9 / 12)
    iou = r["iou"]
    assert iou.dtype == torch.float64 and iou.shape == (3,)
    assert math.isclose(float(iou[0]), 5 / (6 + 7 - 5)) and math.isclose(float(iou[1]), 4 / (6 + 5 - 4))
    assert math.isnan(float(iou[2]))
    assert math.isclose(r["miou"], (5 / 8 + 4 / 7) / 2)
    assert torch.equal(r["confusion"], torch.tensor([[5, 1, 0], [2, 4, 0], [0, 0, 0]]))


def test_predicted_but_absent_class_has_zero_iou():
    r = _metrics([[3, 1], [0, 0]], 4, 0, 1.0).compute()
    assert float(r["iou"][1]) == 0.0 and math.isclose(r["miou"], (3 / 4 + 0) / 2)


def test_invalid_labels_or_no_valid_pixel_give_a_nan_loss():
    r = _metrics([[3, 1], [0, 2]], 6, 2, 3.0).compute()
    assert math.isnan(r["loss"]) and r["invalid"] == 2
    assert math.isclose(r["pixel_accuracy"], 5 / 6)           # the valid pixels are still measured
    r = _metrics([[0, 0], [0, 0]], 0, 0, 0.0).compute()
    assert math.isnan(r["loss"]) and math.isnan(r["pixel_accuracy"]) and math.isnan(r["miou"])


def test_reset_and_state_layout():
    m = _metrics([[3, 1], [0, 2]], 6, 2, 3.0)
    assert m.loss_sum.dtype == torch.float64 and m.confusion.dtype == torch.int64
    m.reset()
    r = m.compute()
    assert r["valid"] == 0 and r["invalid"] == 0 and int(r["confusion"].sum()) == 0 and m.loss_sum.item() == 0.0


def test_constructor_rejects_class_counts_outside_1_to_64():
    import pytest
    for c in (0, 65):
        with pytest.raises(ValueError):
            b200seg.SegmentationMetrics(c, device="cpu")


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, q):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        big = 3 * 2 ** 40 + rank                                  # counts beyond f32 / i32 range travel exactly
        m = _metrics([[rank + 1, 2], [3 * rank, big]], 10 + rank, rank, 0.25 + rank)
        m.all_reduce()
        q.put((rank, m.confusion.tolist(), m.counts.tolist(), float(m.loss_sum[0])))
    finally:
        dist.destroy_process_group()


def test_all_reduce_sums_the_state_over_ranks_world2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    want_cm = [[3, 4], [3, 2 * 3 * 2 ** 40 + 1]]
    for _, cm, counts, loss in res:
        assert cm == want_cm
        assert counts == [21, 1]
        assert loss == 1.5


def test_metrics_entry_points_check_arguments_before_any_cuda_call():
    L = _cabi.lib
    p = 4096                                                      # never dereferenced: every check fails first
    assert L.b200seg_seg_metrics(0, _cabi.F32, _cabi.NCHW, 0, p, _cabi.I64, -100, p, p, p, 1, 10, 8, 8, None) < 0
    assert b"null pointer" in L.b200seg_last_error()
    assert L.b200seg_seg_metrics(p, _cabi.F32, _cabi.NCHW, 0, p, _cabi.I64, -100, p, p, p, 1, 65, 8, 8, None) < 0
    assert b"1..64" in L.b200seg_last_error()
    assert L.b200seg_seg_metrics(p, _cabi.F32, _cabi.NCHW, 0, p, _cabi.F32, -100, p, p, p, 1, 10, 8, 8, None) < 0
    assert b"target dtype" in L.b200seg_last_error()
    assert L.b200seg_seg_metrics(p, _cabi.F32, _cabi.NHWC, 8, p, _cabi.U8, 255, p, p, p, 1, 10, 8, 8, None) < 0
    assert b"ldc" in L.b200seg_last_error()
    assert L.b200seg_seg_metrics(p, _cabi.F32, _cabi.NCHW, 0, p, _cabi.I64, -100, p, p, p, 1, 10, 0, 8, None) < 0
    assert b"empty" in L.b200seg_last_error()
    assert L.b200seg_tail_fused_metrics(p, p, p, p, p, p, _cabi.I64, -100, p, p, p, 1, 8, 8, 17, None) < 0
    assert b"C=17" in L.b200seg_last_error()
    assert L.b200seg_tail_fused_metrics(p, p, p, p, p, p + 8, _cabi.I64, -100, p, p, p, 1, 8, 8, 10, None) < 0
    assert b"16-byte aligned" in L.b200seg_last_error()
    assert L.b200seg_tail_fused_metrics(p, p, p, p, p, p, _cabi.BF16, -100, p, p, p, 1, 8, 8, 10, None) < 0
    assert b"int64 or uint8" in L.b200seg_last_error()
    assert L.b200seg_tail_fused_metrics(p, p, p, p, p, p, _cabi.I64, -100, 0, p, p, 1, 8, 8, 10, None) < 0
    assert b"bad pointers" in L.b200seg_last_error()
