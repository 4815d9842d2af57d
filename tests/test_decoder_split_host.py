"""Host side of the decoder without concat buffers: the bf16 eval schedules and the two-source C-ABI entry points (no GPU)."""
import b200seg
from b200seg import _cabi
from b200seg.engine import Step


def _channels(steps):
    """Channel count of every tensor of a schedule, propagated from the conv weights."""
    ch = {"x": 3}
    for s in steps:
        if s.conv is not None:
            ch[s.dst] = s.conv.weight.shape[0]
        elif s.op == "upcat":
            ch[s.dst] = ch[s.res] + ch[s.src]
        else:
            ch[s.dst] = ch[s.src]
    return ch


def _check(model, H, W, want_cs):
    eng = model._get_engine()
    sched = eng._schedule("bf16", "tc", H, W)
    ch = _channels(eng.steps)
    by_dst = {s.dst: s for s in sched}
    readers = lambda name: [t for t in sched if name in (t.src, t.res, t.skip)]   # noqa: E731
    # no concat buffer feeds a 3x3 conv: every upcat of the unsplit schedule is an upsample alone now
    assert not any(s.op == "upcat" for s in sched)
    two = [s for s in sched if s.skip is not None]
    assert [ch[s.skip] for s in two] == want_cs
    for s in two:
        up = by_dst[s.src]
        assert s.op == "dense" and s.taps == 9 and up.op == "upsample" and up.res is None
        assert s.conv.weight.shape[1] == ch[s.skip] + ch[up.src]            # Cs + Cu is the packed weights' Cin
        assert readers(s.src) == [s] and s.name.endswith(".conv.0")
    # the unsplit schedule (fp32 / exact path, training) keeps the concat
    assert [s.op for s in eng._schedule("fp32", "simt", H, W)].count("upcat") == len(want_cs)
    assert [s.name for s in sched if s.op == "upsample"] == [f"up{k}.up" for k in range(1, len(want_cs) + 1)]


def test_mbv2unet_eval_schedule_reads_skip_and_upsample_directly():
    _check(b200seg.MobileNetV2UNet(output_channels=10), 256, 512, [64, 32, 24, 16])


def test_unet_eval_schedule_reads_skip_and_upsample_directly():
    _check(b200seg.UNet(10), 256, 256, [256, 128, 64])


def test_split_keeps_an_upcat_with_other_readers():
    a = Step("upcat", "u", "lo", "cat", res="sk")
    c = Step("dense", "c", "cat", "y", taps=9)
    r = Step("dense", "r", "y", "z", taps=9, res="cat")           # the concat is also a residual: it must exist
    assert b200seg.engine.Engine._split_upcat([a, c, r]) == [a, c, r]
    p = Step("dense", "p", "cat", "y", taps=1)                       # 1x1 reader: not a two-source step
    assert b200seg.engine.Engine._split_upcat([a, p]) == [a, p]
    out = b200seg.engine.Engine._split_upcat([a, c])
    assert out[0].op == "upsample" and out[0].src == "lo" and out[1].skip == "sk" and out[1].src == out[0].dst


def test_two_source_entry_points_validate_before_any_cuda_call():
    lib = _cabi.lib
    rc = lib.b200seg_conv_tc_cat(0, 1, 1, 0, 0, 1, 1, 8, 8, 12, 16, 16, 9, 0, 0, 0)
    assert rc < 0 and b"multiples of 8" in lib.b200seg_last_error()
    rc = lib.b200seg_conv_tc_cat(0, 1, 1, 0, 0, 1, 1, 8, 8, 16, 16, 16, 9, 0, 0, 0)
    assert rc < 0 and b"null pointer" in lib.b200seg_last_error()          # Cs > 0 needs a skip tensor
    rc = lib.b200seg_conv_tc_cat(1, 1, 1, 0, 0, 1, 1, 8, 8, 16, 0, 16, 9, 0, 0, 0)
    assert rc < 0 and b"Cu" in lib.b200seg_last_error()
    rc = lib.b200seg_conv_tc_cat(1, 1, 1, 0, 0, 1, 1, 8, 8, 16, 16, 16, 4, 0, 0, 0)
    assert rc < 0 and b"taps" in lib.b200seg_last_error()
    rc = lib.b200seg_conv_rs_cat(0, 1, 1, 0, 0, 1, 2, 128, 256, 16, 64, 32, 1, 0, 0)
    assert rc < 0 and b"bad arguments" in lib.b200seg_last_error()
    rc = lib.b200seg_conv_rs_cat(1, 1, 1, 0, 0, 1, 2, 64, 128, 24, 128, 64, 1, 0, 0)
    assert rc < 0 and b"unsupported shape" in lib.b200seg_last_error()


def test_conv_rs_cat_supported_agrees_with_the_concat_shape():
    lib = _cabi.lib
    assert lib.b200seg_conv_rs_cat_supported(128, 256, 16, 64, 32) == 1      # MobileNetV2UNet up4.conv.0
    assert lib.b200seg_conv_rs_cat_supported(128, 256, 0, 80, 32) == lib.b200seg_conv_rs_supported(128, 256, 80, 32) == 1
    assert lib.b200seg_conv_rs_cat_supported(64, 128, 24, 128, 64) == 0      # up3.conv.0: 64 output channels
    assert lib.b200seg_conv_rs_cat_supported(128, 256, 12, 64, 32) == 0      # skip channels not a multiple of 8
    assert lib.b200seg_conv_rs_cat_supported(32, 64, 16, 64, 32) == 0        # narrow map
