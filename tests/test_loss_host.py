"""CrossEntropyLoss options without a GPU: constructor validation as torch, the ``weight`` buffer in ``state_dict``, and the
argument checks of the new C entry points (they return before any CUDA call)."""
import warnings

import pytest
import torch

import b200seg
from b200seg import _cabi

lib = _cabi.lib


def test_constructor_defaults_match_torch():
    ours, ref = b200seg.CrossEntropyLoss(), torch.nn.CrossEntropyLoss()
    for k in ("ignore_index", "reduction", "label_smoothing"):
        assert getattr(ours, k) == getattr(ref, k), k
    assert ours.weight is None
    assert list(ours.state_dict()) == list(ref.state_dict()) == []


@pytest.mark.parametrize("reduction", ["mean", "sum", "none"])
def test_constructor_takes_torch_arguments(reduction):
    w = torch.rand(5) + 0.5
    m = b200seg.CrossEntropyLoss(weight=w, ignore_index=255, reduction=reduction, label_smoothing=0.1)
    assert m.reduction == reduction and m.ignore_index == 255 and m.label_smoothing == pytest.approx(0.1)
    assert torch.equal(m.weight, w)
    assert "weight" in dict(m.named_buffers())


def test_constructor_rejects_what_torch_rejects():
    with pytest.raises(ValueError, match="not a valid value for reduction"):
        b200seg.CrossEntropyLoss(reduction="avg")
    for bad in (-0.1, 1.5):
        with pytest.raises(RuntimeError, match="label_smoothing must be between 0.0 and 1.0"):
            b200seg.CrossEntropyLoss(label_smoothing=bad)
    with pytest.raises(ValueError, match="1-D"):
        b200seg.CrossEntropyLoss(weight=torch.ones(2, 5))
    b200seg.CrossEntropyLoss(label_smoothing=0.0)
    b200seg.CrossEntropyLoss(label_smoothing=1.0)


@pytest.mark.parametrize("size_average,reduce,want", [(None, False, "none"), (False, None, "sum"), (True, True, "mean"),
                                                      (False, False, "none")])
def test_legacy_size_average_and_reduce_map_like_torch(size_average, reduce, want):
    with warnings.catch_warnings(record=True) as got:
        warnings.simplefilter("always")
        m = b200seg.CrossEntropyLoss(size_average=size_average, reduce=reduce)
        ref = torch.nn.CrossEntropyLoss(size_average=size_average, reduce=reduce)
    assert m.reduction == ref.reduction == want
    assert any("size_average and reduce args will be deprecated" in str(w.message) for w in got)


def test_weight_buffer_round_trips_with_torch_state_dict():
    w = torch.tensor([0.5, 2.0, 1.0, 0.0, 3.0])
    ref = torch.nn.CrossEntropyLoss(weight=w)
    ours = b200seg.CrossEntropyLoss(weight=torch.ones(5))
    ours.load_state_dict(ref.state_dict())
    assert list(ours.state_dict()) == ["weight"]
    assert torch.equal(ours.weight, w)
    back = torch.nn.CrossEntropyLoss(weight=torch.zeros(5))
    back.load_state_dict(ours.state_dict())
    assert torch.equal(back.weight, w)
    with pytest.raises(RuntimeError, match="Unexpected key"):
        b200seg.CrossEntropyLoss().load_state_dict(ref.state_dict())


def test_forward_on_cpu_is_an_error():
    m = b200seg.CrossEntropyLoss(weight=torch.ones(3), label_smoothing=0.1)
    with pytest.raises(RuntimeError, match="CUDA only"):
        m(torch.zeros(1, 3, 4, 4), torch.zeros(1, 4, 4, dtype=torch.uint8))


def _err():
    return lib.b200seg_last_error().decode()


P = 1 << 12      # a non-null pointer value; never dereferenced, the checks return first


def test_softmax_ce_ex_rejects_bad_arguments_before_any_cuda_call():
    def call(logits=P, target=P, tdt=_cabi.I64, ls=0.0, loss_sum=P, loss_map=None, dl=None, denom=None, B=1, C=3, H=4, W=4):
        return lib.b200seg_softmax_ce_ex(logits, target, tdt, -100, None, ls, loss_sum, loss_map, dl, denom, B, C, H, W, None)

    cases = [
        (dict(C=0), "C=0"),
        (dict(H=0), "empty"),
        (dict(logits=None), "null"),
        (dict(target=None), "null"),
        (dict(tdt=_cabi.F32), "target_dtype"),
        (dict(tdt=7), "target_dtype"),
        (dict(ls=1.5), "label_smoothing"),
        (dict(ls=-0.25), "label_smoothing"),
        (dict(ls=float("nan")), "label_smoothing"),
        (dict(loss_sum=None), "exactly one"),
        (dict(loss_map=P), "exactly one"),
        (dict(loss_sum=None, loss_map=P, dl=P), "no gradient"),
        (dict(loss_sum=None, loss_map=P, denom=P), "denom"),
    ]
    for kw, msg in cases:
        rc = call(**kw)
        assert rc < 0, kw
        assert msg in _err(), (kw, _err())


def test_softmax_ce_ex_bwd_and_count_reject_bad_arguments():
    rc = lib.b200seg_softmax_ce_ex_bwd(P, P, _cabi.U8, 255, None, 0.1, None, P, 1, 3, 4, 4, None)
    assert rc < 0 and "null gout" in _err()
    rc = lib.b200seg_softmax_ce_ex_bwd(P, P, _cabi.U8, 255, None, 0.1, P, None, 1, 3, 4, 4, None)
    assert rc < 0 and "dlogits" in _err()
    rc = lib.b200seg_softmax_ce_ex_bwd(P, P, _cabi.BF16, 255, None, 0.1, P, P, 1, 3, 4, 4, None)
    assert rc < 0 and "target_dtype" in _err()
    rc = lib.b200seg_softmax_ce_ex_bwd(P, P, _cabi.I64, -100, None, 2.0, P, P, 1, 3, 4, 4, None)
    assert rc < 0 and "label_smoothing" in _err()
    rc = lib.b200seg_ce_count_ex(None, _cabi.I64, -100, None, P, 16, 3, None)
    assert rc < 0 and "ce_count_ex" in _err()
    rc = lib.b200seg_ce_count_ex(P, _cabi.I64, -100, None, P, 0, 3, None)
    assert rc < 0 and "ce_count_ex" in _err()
    rc = lib.b200seg_ce_count_ex(P, 9, -100, None, P, 16, 3, None)
    assert rc < 0 and "target_dtype" in _err()
