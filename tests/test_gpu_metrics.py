"""Validation metrics on the GPU (b200seg.SegmentationMetrics, model.evaluate): the standalone kernel against torch, the
metrics epilogue of the fused output tail against predict_mask and the logits-mode tail, the UNet / fp32 / C > 16 paths,
a trained network against the fp32 oracle, CUDA-graph capture, and argument errors."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

import b200seg  # noqa: E402
from b200seg import ops  # noqa: E402
from oracle import unet_oracle as O  # noqa: E402
from util import expand_aliases, f2_meta, f2_sd, fixture_sd  # noqa: E402

DEV = "cuda"


def _targets(B, H, W, C, seed, ignore=-100, n_ignore=0.1, dtype=torch.int64):
    g = torch.Generator().manual_seed(seed)
    t = torch.randint(0, C, (B, H, W), generator=g)
    t[torch.rand(B, H, W, generator=g) < n_ignore] = ignore
    return t.to(dtype).to(DEV)


def _ref(logits, t, C, ignore):
    """torch: confusion by bincount of the argmax over the counted pixels, counts, and the f64 cross-entropy sum
    (F.cross_entropy(ignore_index=ignore) when ``ignore`` is a class index)."""
    t64 = t.long()
    valid = (t64 >= 0) & (t64 < C) & (t64 != ignore)
    invalid = ((t64 < 0) | (t64 >= C)) & (t64 != ignore)
    pred = logits.argmax(1)
    cm = torch.bincount(t64[valid] * C + pred[valid], minlength=C * C).view(C, C)
    if 0 <= ignore < C:       # every pixel that is not counted carries the ignore label (torch asserts on out-of-range ones)
        tt = torch.where(valid, t64, torch.full_like(t64, ignore))
        loss = F.cross_entropy(logits.double(), tt, ignore_index=ignore, reduction="sum")
    else:
        tt = torch.where(valid, t64, torch.full_like(t64, -12345))
        loss = F.cross_entropy(logits.double(), tt, ignore_index=-12345, reduction="sum")
    return cm.cpu(), int(valid.sum()), int(invalid.sum()), float(loss)


def _state(m):
    return m.confusion.cpu(), int(m.counts[0]), int(m.counts[1]), float(m.loss_sum[0])


def _assert_matches(m, ref, rtol=1e-5):
    cm, nv, ni, loss = _state(m)
    rcm, rnv, rni, rloss = ref
    assert torch.equal(cm, rcm), (cm, rcm)
    assert (nv, ni) == (rnv, rni)
    assert abs(loss - rloss) <= rtol * max(abs(rloss), 1e-30), (loss, rloss)


# ------------------------------------------------------------------------------------------ 1. standalone kernel vs torch
@pytest.mark.parametrize("C", [1, 10, 16, 19, 40])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shape", [(3, 64, 96), (2, 37, 53), (1, 6, 7)])
@pytest.mark.parametrize("tkind", ["i64", "u8"])
def test_standalone_kernel_matches_torch(C, dtype, shape, tkind):
    B, H, W = shape
    g = torch.Generator().manual_seed(C * 100 + H)
    logits = (torch.randn(B, C, H, W, generator=g) * 3).to(dtype).to(DEV)
    ignore = -100 if tkind == "i64" else 255
    t = _targets(B, H, W, C, seed=H + C, ignore=ignore, dtype=torch.int64 if tkind == "i64" else torch.uint8)
    m = b200seg.SegmentationMetrics(C, device=DEV, ignore_index=ignore)
    m.update(logits, t)
    _assert_matches(m, _ref(logits, t, C, ignore))


def test_first_maximum_wins_on_ties():
    C, B, H, W = 10, 2, 32, 64
    g = torch.Generator().manual_seed(5)
    for dtype in (torch.float32, torch.bfloat16):
        logits = torch.randint(0, 3, (B, C, H, W), generator=g).to(dtype).to(DEV)      # ties everywhere
        t = _targets(B, H, W, C, seed=6)
        m = b200seg.SegmentationMetrics(C, device=DEV)
        m.update(logits, t)
        _assert_matches(m, _ref(logits, t, C, -100))
        # odd W: the one-pixel kernel follows the same rule
        m.reset().update(logits[..., :63].contiguous(), t[..., :63].contiguous())
        _assert_matches(m, _ref(logits[..., :63], t[..., :63], C, -100))


def test_out_of_range_labels_are_invalid_and_make_the_loss_nan():
    C = 10
    logits = torch.randn(2, C, 16, 32, device=DEV)
    t = _targets(2, 16, 32, C, seed=1)
    t[0, 0, :5] = 10
    t[1, 3, 7] = 77
    t[1, 4, 8] = -1
    m = b200seg.SegmentationMetrics(C, device=DEV)
    m.update(logits, t)
    _assert_matches(m, _ref(logits, t, C, -100))
    r = m.compute()
    assert r["invalid"] == 7
    assert r["loss"] != r["loss"]                    # NaN, like b200seg.CrossEntropyLoss on such a batch
    assert r["miou"] == r["miou"]                    # the confusion of the valid pixels is still reported


@pytest.mark.parametrize("ignore", [0, 3])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shape", [(2, 64, 96), (2, 37, 53)])
@pytest.mark.parametrize("tkind", ["i64", "u8"])
def test_ignore_index_inside_the_class_range(ignore, dtype, shape, tkind):
    """ignore_index may be a class index: those pixels contribute nothing, as with F.cross_entropy(ignore_index=k)."""
    C, (B, H, W) = 10, shape
    g = torch.Generator().manual_seed(17)
    logits = (torch.randn(B, C, H, W, generator=g) * 3).to(dtype).to(DEV)
    t = _targets(B, H, W, C, seed=18, n_ignore=0.0, dtype=torch.int64 if tkind == "i64" else torch.uint8)
    m = b200seg.SegmentationMetrics(C, device=DEV, ignore_index=ignore).update(logits, t)
    ref = _ref(logits, t, C, ignore)
    _assert_matches(m, ref)
    keep = t.long() != ignore
    assert ref[1] == int(keep.sum()) and int(ref[0][ignore].sum()) == 0
    assert torch.equal(ref[0], torch.bincount(t.long()[keep] * C + logits.argmax(1)[keep], minlength=C * C).view(C, C).cpu())


def test_minus_inf_logits_give_torch_cross_entropy():
    """Classes masked with -inf (also the first ones of a pixel) add nothing to the log-sum-exp instead of a NaN."""
    C, B, H, W = 10, 2, 16, 32
    for shape_w in (W, 31):                                     # 4-pixel and one-pixel kernels
        logits = torch.randn(B, C, H, shape_w, device=DEV) * 3
        logits[:, :3] = float("-inf")                           # the first classes of every pixel
        logits[0, 5, :4] = float("-inf")
        t = _targets(B, H, shape_w, C, seed=21)
        t[(t >= 0) & (t < 3)] = 4                               # targets on finite logits: a finite loss
        t0 = t[0, :4]
        t0[t0 == 5] = 4
        m = b200seg.SegmentationMetrics(C, device=DEV).update(logits, t)
        ref = _ref(logits, t, C, -100)
        assert ref[3] == ref[3] and abs(ref[3]) != float("inf")
        _assert_matches(m, ref)


def test_non_contiguous_and_offset_targets_are_copied():
    C, B, H, W = 10, 2, 64, 96
    logits = torch.randn(B, C, H, W, device=DEV)
    big = _targets(B, H, W + 8, C, seed=23)
    t = big[:, :, 3:3 + W]                                       # a crop: neither contiguous nor aligned
    assert not t.is_contiguous()
    m = b200seg.SegmentationMetrics(C, device=DEV).update(logits, t)
    _assert_matches(m, _ref(logits, t.contiguous(), C, -100))
    model = _mb(C)
    x = O.synth_input(B, H, W, seed=24).to(DEV)
    a = model.evaluate(x, t, b200seg.SegmentationMetrics(C, device=DEV))
    b = model.evaluate(x, t.contiguous(), b200seg.SegmentationMetrics(C, device=DEV))
    sa, sb = _state(a), _state(b)
    assert torch.equal(sa[0], sb[0]) and sa[1:3] == sb[1:3]
    assert abs(sa[3] - sb[3]) <= 1e-9 * sb[3]


# ------------------------------------------------------------------------------------------ 2. fused tail (MobileNetV2UNet bf16)
def _mb(C, precision="bf16"):
    m = b200seg.MobileNetV2UNet(output_channels=C)
    m.load_state_dict(expand_aliases(fixture_sd(C)), strict=True)
    m = m.to(DEV).eval()
    m._get_engine().precision = precision
    return m


@pytest.mark.parametrize("C", [1, 10, 16, 19])
@pytest.mark.parametrize("shape", [(2, 64, 96), (1, 160, 288)])
def test_evaluate_matches_predict_mask_and_logits(C, shape):
    """C <= 16: the metrics epilogue of the fused tail; C = 19: the upsample + standalone kernel fallback.  The confusion
    equals the histogram of predict_mask exactly, the loss the cross-entropy of the logits-mode output."""
    B, H, W = shape
    m = _mb(C)
    eng = m._get_engine()
    x = O.synth_input(B, H, W, seed=3).to(DEV)
    t = _targets(B, H, W, C, seed=4)
    with torch.no_grad():
        logits = m(x)                                   # f32 NCHW logits of the same tail arithmetic
        mask = m.predict_mask(x)
    ref = _ref(logits, t, C, -100)
    valid = (t >= 0) & (t < C)
    assert torch.equal(ref[0], torch.bincount(t[valid] * C + mask.long()[valid], minlength=C * C).view(C, C).cpu())
    met = b200seg.SegmentationMetrics(C, device=DEV)
    for _ in range(4):                                  # the later calls replay the captured graph
        met.reset()
        assert m.evaluate(x, t, met) is met
        _assert_matches(met, ref)
    assert any(e["graph"] is not None for e in eng._graphs.values()), "graph was never captured"
    # ignore_index inside the class range (C > 1): those pixels drop out of the fused epilogue too
    if C > 1:
        mi = b200seg.SegmentationMetrics(C, device=DEV, ignore_index=C - 1)
        m.evaluate(x, t, mi)
        _assert_matches(mi, _ref(logits, t, C, C - 1))
    # uint8 targets with 255 as the ignore label: the same result
    t8 = torch.where(valid, t, torch.full_like(t, 255)).to(torch.uint8)
    met8 = b200seg.SegmentationMetrics(C, device=DEV, ignore_index=255)
    m.evaluate(x, t8, met8)
    _assert_matches(met8, ref)
    # two batches accumulate to the sum of their separate results
    x2, t2 = O.synth_input(B, H, W, seed=8).to(DEV), _targets(B, H, W, C, seed=9)
    a = _state(m.evaluate(x2, t2, b200seg.SegmentationMetrics(C, device=DEV)))
    both = b200seg.SegmentationMetrics(C, device=DEV)
    m.evaluate(x, t, both)
    m.evaluate(x2, t2, both)
    cm, nv, ni, loss = _state(both)
    assert torch.equal(cm, ref[0] + a[0]) and nv == ref[1] + a[1] and ni == ref[2] + a[2]
    assert abs(loss - (_state(met)[3] + a[3])) <= 1e-9 * loss


def test_fused_tail_metrics_is_the_tail_that_runs():
    """bf16 MobileNetV2UNet with C <= 16 takes the metrics in the output-tail kernel itself."""
    m = _mb(10)
    steps = m._get_engine()._schedule("bf16", "tc", 64, 96, torch.float32)
    assert steps[-1].op == "tail"


# ------------------------------------------------------------------------------------------ 3. UNet (NHWC) and the fp32 path
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_unet_evaluate_equals_forward_plus_update(precision):
    torch.manual_seed(0)
    m = b200seg.UNet(output_channels=10, base_filters=16).to(DEV).eval()
    m._get_engine().precision = precision
    x = O.synth_input(2, 64, 96, seed=1).to(DEV)
    t = _targets(2, 64, 96, 10, seed=2)
    with torch.no_grad():
        logits = m(x)
        mask = m.predict_mask(x)
    a = b200seg.SegmentationMetrics(10, device=DEV)
    for _ in range(4):
        a.reset()
        m.evaluate(x, t, a)
    b = b200seg.SegmentationMetrics(10, device=DEV).update(logits, t)
    cm, nv, ni, loss = _state(a)
    cm2, nv2, ni2, loss2 = _state(b)
    assert torch.equal(cm, cm2) and (nv, ni) == (nv2, ni2)
    assert abs(loss - loss2) <= 1e-6 * loss2
    valid = (t >= 0) & (t < 10)
    assert torch.equal(cm, torch.bincount(t[valid] * 10 + mask.long()[valid], minlength=100).view(10, 10).cpu())
    _assert_matches(a, _ref(logits, t, 10, -100))


def test_mbv2unet_fp32_evaluate_equals_forward_plus_update():
    m = _mb(10, precision=None)
    x = O.synth_input(2, 64, 96, seed=5).to(DEV)
    t = _targets(2, 64, 96, 10, seed=6)
    with torch.no_grad():
        logits = m(x)
        mask = m.predict_mask(x)
    a = b200seg.SegmentationMetrics(10, device=DEV)
    for _ in range(4):
        a.reset()
        m.evaluate(x, t, a)
    _assert_matches(a, _ref(logits, t, 10, -100))
    valid = (t >= 0) & (t < 10)
    assert torch.equal(_state(a)[0], torch.bincount(t[valid] * 10 + mask.long()[valid], minlength=100).view(10, 10).cpu())


# ------------------------------------------------------------------------------------------ 4. a trained network
def _miou(cm):
    cm = cm.double()
    tp = cm.diagonal()
    union = cm.sum(0) + cm.sum(1) - tp
    iou = tp[union > 0] / union[union > 0]
    return float(iou.mean())


def test_f2_bf16_miou_matches_the_fp32_oracle():
    sd, meta = f2_sd(), f2_meta()["full"]
    b, h, w = meta["shape"]
    x, t = O.road_scene_batch(b, h, w, seed=meta["seed"])
    with torch.no_grad():
        ref = O.mobilenetv2_unet_forward(sd, x)
    cm_ref = torch.bincount(t.reshape(-1) * 10 + ref.argmax(1).reshape(-1), minlength=100).view(10, 10)
    m = b200seg.MobileNetV2UNet(output_channels=10)
    full = dict(m.state_dict())
    full.update(expand_aliases(sd))
    m.load_state_dict(full, strict=True)
    m = m.to(DEV).bfloat16().eval()
    met = b200seg.SegmentationMetrics(10, device=DEV)
    m.evaluate(x.to(DEV).bfloat16(), t.to(DEV), met)
    r = met.compute()
    assert r["valid"] == t.numel() and r["invalid"] == 0
    assert abs(r["miou"] - _miou(cm_ref)) < 0.002, (r["miou"], _miou(cm_ref))
    assert r["miou"] > 0.5                           # a trained network, not a constant predictor
    assert abs(r["loss"] - float(F.cross_entropy(ref.double(), t))) < 0.05 * float(F.cross_entropy(ref.double(), t)) + 1e-3


# ------------------------------------------------------------------------------------------ 5. capture
def test_update_is_capturable_in_a_cuda_graph():
    C = 10
    logits = torch.randn(2, C, 64, 96, device=DEV)
    t = _targets(2, 64, 96, C, seed=11)
    met = b200seg.SegmentationMetrics(C, device=DEV)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        met.update(logits, t)                         # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    met.reset()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        met.update(logits, t)
    met.reset()
    g.replay()
    g.replay()
    cm, nv, ni, loss = _ref(logits, t, C, -100)
    _assert_matches(met, (2 * cm, 2 * nv, 2 * ni, 2 * loss))


# ------------------------------------------------------------------------------------------ 6. errors
def test_argument_errors():
    m = _mb(10)
    x = O.synth_input(2, 64, 96, seed=0).to(DEV)
    t = _targets(2, 64, 96, 10, seed=0)
    met = b200seg.SegmentationMetrics(10, device=DEV)
    m.train()
    with pytest.raises(RuntimeError, match="eval"):
        m.evaluate(x, t, met)
    m.eval()
    with pytest.raises(RuntimeError):
        m.evaluate(x.cpu(), t.cpu(), met)
    with pytest.raises(RuntimeError):
        met.update(torch.randn(2, 10, 64, 96), t.cpu())
    with pytest.raises(ValueError):
        m.evaluate(x, t[:, :, :64], met)                                          # shape
    with pytest.raises(ValueError):
        m.evaluate(x, t[:1], met)
    with pytest.raises(ValueError):
        m.evaluate(x, t, b200seg.SegmentationMetrics(5, device=DEV))              # class count
    with pytest.raises(ValueError):
        m.evaluate(x, t.int(), met)                                               # dtype
    with pytest.raises(ValueError):
        met.update(torch.randn(2, 10, 64, 96, device=DEV), t.float())
    with pytest.raises(ValueError):
        met.update(torch.randn(2, 5, 64, 96, device=DEV), t)
    with pytest.raises(ValueError):
        met.update(torch.randn(2, 10, 64, 96, device=DEV).half(), t)
    with pytest.raises(ValueError):
        b200seg.SegmentationMetrics(65, device=DEV)
    big = b200seg.SegmentationMetrics(64, device=DEV)
    with pytest.raises(RuntimeError, match="64"):                                 # the kernel's own limit
        ops.seg_metrics(torch.randn(1, 65, 8, 8, device=DEV), torch.zeros(1, 8, 8, dtype=torch.int64, device=DEV), 65, -100,
                        big.confusion, big.counts, big.loss_sum)
    assert int(met.counts.sum()) == 0 and int(big.counts.sum()) == 0
