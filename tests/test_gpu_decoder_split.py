"""Decoder convolutions on two sources: conv_tc / conv_rs read cat([skip, up], channel) from the two dense tensors instead
of a concat buffer, and the upsample step writes only the upsampled half.

Bit-identity is required wherever the sequence of issued K = 16 groups is the concat path's: Cs a multiple of 64 in any
mode, and Cs a multiple of 16 in TAP mode (maps narrower than 96 columns, or flags bit1), whose loop is tap-major.  HALO
mode and conv_rs loop chunk-major, so a skip chunk narrower than 64 channels changes the fp32 accumulation order there:
those cases are checked against the float64 reference with test_gpu_ops' tolerance and against the concat path within one
bf16 ulp of the largest output.
"""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

import b200seg  # noqa: E402
from b200seg import ops  # noqa: E402
from b200seg._cabi import lib  # noqa: E402

DEV = "cuda"
TOL_BF16 = 6e-3          # test_gpu_ops: fp32 accumulation order + one bf16 output rounding, relative to the output range


def _err(got, ref):
    got, ref = got.double(), ref.double()
    return float((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


def _nchw(t):
    return t.permute(0, 3, 1, 2).contiguous()


def _rand(*shape, seed=0, scale=1.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(DEV)


def _operands(B, H, W, Cs, Cu, Cout, seed):
    s = _rand(B, Cs, H, W, seed=seed).bfloat16()
    u = _rand(B, Cu, H, W, seed=seed + 1).bfloat16()
    w = _rand(Cout, Cs + Cu, 3, 3, seed=seed + 2, scale=(2.0 / ((Cs + Cu) * 9)) ** 0.5).bfloat16()
    b = _rand(Cout, seed=seed + 3, scale=0.1)
    return s, u, w, b


def _same_k_groups(W, Cs, flags, rs):
    halo = W >= 96 and not (flags & 2)
    return Cs % 64 == 0 or (Cs % 16 == 0 and not halo and not rs)


# MobileNetV2UNet decoder stages at 256 x 512 (Cs + Cu -> Cout at H x W), the plain UNet's whole-chunk skips, ragged tails
TC_CASES = [  # B, H, W, Cs, Cu, Cout
    (2, 16, 32, 64, 1280, 256),      # up1.conv.0: TAP, 21 chunks, MPAIR 2 (streamed weights)
    (2, 32, 64, 32, 256, 128),       # up2.conv.0: TAP, narrow skip chunk (2 k-steps)
    (2, 64, 128, 24, 128, 64),       # up3.conv.0: HALO, 24-channel skip chunk
    (2, 128, 256, 16, 64, 64),       # up4 shape with 64 output channels: HALO on conv_tc, resident weights
    (1, 32, 128, 128, 256, 128),     # UNet up2-like: whole-chunk skip, HALO
    (1, 64, 96, 256, 256, 64),       # UNet up1-like at W = 96: HALO boundary
    (2, 9, 40, 64, 72, 40),          # ragged U tail (8 channels), ragged N
    (1, 7, 130, 24, 40, 32),         # narrow skip + ragged U tail, HALO with a ragged column tile
    (1, 5, 33, 16, 8, 16),           # tiny: one k-step per source
]
FLAGS = [0, 2, 4, 32, 4 | 32, 2 | 4]       # auto, TAP forced, streamed weights, no M pairing, both, TAP + streamed


@pytest.mark.parametrize("flags", FLAGS, ids=["auto", "tap", "streamed", "mpair1", "streamed_mpair1", "tap_streamed"])
@pytest.mark.parametrize("B,H,W,Cs,Cu,Cout", TC_CASES)
def test_conv_tc_two_sources_match_concat(flags, B, H, W, Cs, Cu, Cout):
    s, u, w, b = _operands(B, H, W, Cs, Cu, Cout, seed=31)
    wk = w.permute(0, 2, 3, 1).reshape(Cout, -1).contiguous()
    cat = _nhwc(torch.cat([s, u], 1))
    flags |= 1 << 6      # an unused bit: never dispatched to conv_rs, so every case runs conv_tc
    got = ops.conv_tc(_nhwc(u), wk, b, 9, 1, flags=flags, skip=_nhwc(s))
    old = ops.conv_tc(cat, wk, b, 9, 1, flags=flags)
    torch.cuda.synchronize()
    if _same_k_groups(W, Cs, flags, rs=False):
        assert torch.equal(got, old)
    else:
        ref = F.relu(F.conv2d(torch.cat([s, u], 1).double(), w.double(), b.double(), 1, 1))
        assert _err(_nchw(got), ref) < TOL_BF16
        assert _err(got.float(), old.double()) < 8e-3          # one bf16 ulp of the largest output
    again = ops.conv_tc(_nhwc(u), wk, b, 9, 1, flags=flags, skip=_nhwc(s))
    assert torch.equal(got, again)                              # no atomics: bit-repeatable


RS_CASES = [  # B, H, W, Cs, Cu, Cout, res
    (2, 128, 256, 16, 64, 32, False),    # up4.conv.0
    (2, 40, 256, 64, 64, 32, False),     # whole skip chunk: same K-group order as the concat
    (1, 9, 150, 24, 40, 16, True),       # narrow skip, ragged U tail and column tile, 16-column variant, residual
    (1, 5, 130, 8, 24, 8, False),        # one k-step per source
]


@pytest.mark.parametrize("flags", [0, 1 << 20], ids=["auto", "1cta"])
@pytest.mark.parametrize("B,H,W,Cs,Cu,Cout,res", RS_CASES)
def test_conv_rs_two_sources_match_concat(flags, B, H, W, Cs, Cu, Cout, res):
    assert lib.b200seg_conv_rs_cat_supported(H, W, Cs, Cu, Cout) == 1
    s, u, w, b = _operands(B, H, W, Cs, Cu, Cout, seed=41)
    r = _rand(B, Cout, H, W, seed=45).bfloat16() if res else None
    wk = w.permute(0, 2, 3, 1).reshape(Cout, -1).contiguous()
    rr = _nhwc(r) if res else None
    got = ops.conv_rs(_nhwc(u), wk, b, 1, rr, flags=flags, skip=_nhwc(s))
    old = ops.conv_rs(_nhwc(torch.cat([s, u], 1)), wk, b, 1, rr, flags=flags)
    torch.cuda.synchronize()
    if flags == 0:
        assert torch.equal(got, ops.conv_tc(_nhwc(u), wk, b, 9, 1, rr, skip=_nhwc(s)))   # conv_tc dispatches this shape here
    if _same_k_groups(W, Cs, flags, rs=True):
        assert torch.equal(got, old)
    else:
        ref = F.relu(F.conv2d(torch.cat([s, u], 1).double(), w.double(), b.double(), 1, 1))
        if res:
            ref = ref + r.double()
        assert _err(_nchw(got), ref) < TOL_BF16
        assert _err(got.float(), old.double()) < 8e-3


@pytest.mark.parametrize("B,h,w,Cs,Cu", [(2, 8, 16, 64, 1280), (2, 16, 32, 32, 256), (2, 32, 64, 24, 128),
                                         (2, 64, 128, 16, 64), (1, 3, 5, 8, 16), (2, 4, 9, 16, 24), (1, 1, 1, 8, 8)])
def test_upsample_alone_is_the_concat_kernels_up_slice(B, h, w, Cs, Cu):
    x = _nhwc(_rand(B, Cu, h, w, seed=51).bfloat16())
    skip = _nhwc(_rand(B, Cs, 2 * h, 2 * w, seed=52).bfloat16())
    up = ops.upsample2x_concat(None, x)
    cat = ops.upsample2x_concat(skip, x)
    assert up.shape == (B, 2 * h, 2 * w, Cu)
    assert torch.equal(up, cat[..., Cs:])


@pytest.mark.parametrize("arch", ["mbv2unet", "unet"])
def test_split_schedule_matches_concat_steps_on_the_same_inputs(arch):
    """Each decoder stage of the bf16 eval schedule against the parent's two steps (upsample + concat, conv on the concat
    buffer) on identical inputs: bit-identical for whole-chunk skips and TAP-mode stages, within one bf16 ulp elsewhere
    (MobileNetV2UNet up3 and up4 at this size: HALO / conv_rs with 24- and 16-channel skips)."""
    torch.manual_seed(0)
    m = b200seg.MobileNetV2UNet(output_channels=10) if arch == "mbv2unet" else b200seg.UNet(10)
    m = m.to(DEV).eval()
    eng = m._get_engine()
    eng.precision = "bf16"
    H, W = 256, 512 if arch == "mbv2unet" else 256
    x = torch.randn(2, 3, H, W, device=DEV)
    keep = {}
    with torch.no_grad():
        eng.forward_eval(x, keep=keep)
    pk = eng._pack_eval("bf16")
    sched = eng._schedule("bf16", "tc", H, W, x.dtype)
    two = [s for s in sched if s.skip is not None]
    assert len(two) == (4 if arch == "mbv2unet" else 3)
    for st in two:
        cat = ops.upsample2x_concat(keep[st.skip], keep[[u for u in sched if u.dst == st.src][0].src])
        p = pk[st.name]
        old = ops.conv_tc(cat, p["w"], p["b"], 9, st.act)
        got = keep[st.dst]
        Wst = got.shape[2]
        Cs = keep[st.skip].shape[-1]
        rs = bool(lib.b200seg_conv_rs_supported(got.shape[1], Wst, cat.shape[-1], got.shape[-1]))
        if _same_k_groups(Wst, Cs, 0, rs):
            assert torch.equal(got, old), st.name
        else:
            assert _err(got.float(), old.double()) < 8e-3, st.name
