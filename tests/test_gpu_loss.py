"""b200seg.CrossEntropyLoss with torch's arguments (weight, ignore_index, reduction, label_smoothing) and uint8 targets,
against torch.nn.functional.cross_entropy in float64 on the same f32 logits.  The class counts reach every kernel path: the
4-pixel vector kernels (C <= 16 and H*W % 4 == 0), the one-pixel register kernels (C <= 32) and the any-C kernel."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

import b200seg  # noqa: E402
from oracle import unet_oracle as O  # noqa: E402
from util import expand_aliases, f2_sd  # noqa: E402

DEV = "cuda"

# (ignore_index, target dtype)
TARGETS = [(-100, torch.int64), (0, torch.int64), (3, torch.int64), (-100, torch.uint8), (3, torch.uint8), (255, torch.uint8)]


def _weight(kind, C, g):
    if kind is None:
        return None
    w = torch.rand(C, generator=g, dtype=torch.float64) * 2.0 + 0.25
    if kind == "zeros":
        w[1::2] = 0.0                  # odd classes weigh nothing (C = 1 keeps its one weighted class)
    return w.float()


def _case(B, C, H, W, ignore_index, tdt, seed):
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(B, C, H, W, generator=g) * 3.0
    t = torch.randint(0, C, (B, H, W), generator=g)
    if tdt == torch.int64 or 0 <= ignore_index <= 255:        # a uint8 label cannot be -100
        t[torch.rand(B, H, W, generator=g) < 0.15] = ignore_index
    return z, t.to(tdt), g


def _ref(z, t, w, ignore_index, ls, red, gout=None, scale=3.0):
    z64 = z.double().to(DEV).requires_grad_()
    loss = F.cross_entropy(z64, t.long().to(DEV), weight=None if w is None else w.double().to(DEV), ignore_index=ignore_index,
                           reduction=red, label_smoothing=ls)
    (loss * scale).backward() if gout is None else (loss * gout.double()).sum().backward()
    return loss.detach(), z64.grad


def _rel(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))


@pytest.mark.parametrize("red", ["mean", "sum", "none"])
@pytest.mark.parametrize("ls", [0.0, 0.1, 1.0])
@pytest.mark.parametrize("wkind", [None, "random", "zeros"])
@pytest.mark.parametrize("hw", [(8, 12), (7, 9)])
@pytest.mark.parametrize("C", [1, 3, 10, 16, 24, 40])
def test_matches_torch_cross_entropy(C, hw, wkind, ls, red):
    H, W = hw
    for k, (ignore_index, tdt) in enumerate(TARGETS):
        z, t, g = _case(2, C, H, W, ignore_index, tdt, seed=1000 * C + 10 * H + k)
        w = _weight(wkind, C, g)
        crit = b200seg.CrossEntropyLoss(weight=w, ignore_index=ignore_index, reduction=red, label_smoothing=ls).to(DEV)
        zd = z.to(DEV).requires_grad_()
        loss = crit(zd, t.to(DEV))
        gout = None
        if red == "none":
            gout = torch.randn(2, H, W, generator=g).to(DEV)
            loss.backward(gout)
        else:
            (loss * 3).backward()
        ref, gref = _ref(z, t, w, ignore_index, ls, red, gout)
        what = (C, hw, wkind, ls, red, ignore_index, tdt)
        assert loss.dtype == torch.float32 and loss.shape == ref.shape, what
        if red == "none":
            assert _rel(loss, ref) <= 1e-5, what
        elif math.isnan(float(ref)):          # every pixel ignored (ignore_index 0 with C = 1): NaN, as torch
            assert math.isnan(float(loss)), what
            continue
        else:
            assert abs(float(loss) - float(ref)) <= 1e-5 * abs(float(ref)), (what, float(loss), float(ref))
        assert _rel(zd.grad, gref) <= 1e-6, (what, _rel(zd.grad, gref))


@pytest.mark.parametrize("C,hw", [(5, (8, 8)), (5, (7, 9)), (24, (8, 8)), (40, (8, 8))])
@pytest.mark.parametrize("tdt", [torch.int64, torch.uint8])
def test_bad_labels_give_nan(C, hw, tdt):
    H, W = hw
    ii = 255 if tdt == torch.uint8 else -100
    z, t, _ = _case(2, C, H, W, ii, tdt, seed=7)
    t[0, 1, 2] = C + 2                                           # neither a class nor ignore_index
    w = torch.rand(C) + 0.5
    for red in ("mean", "sum"):
        zd = z.to(DEV).requires_grad_()
        loss = b200seg.CrossEntropyLoss(weight=w.to(DEV), ignore_index=ii, reduction=red, label_smoothing=0.1)(zd, t.to(DEV))
        assert torch.isnan(loss), red
        loss.backward()
        assert torch.isfinite(zd.grad).all() and float(zd.grad[0, :, 1, 2].abs().max()) == 0.0
    zd = z.to(DEV).requires_grad_()
    m = b200seg.CrossEntropyLoss(ignore_index=ii, reduction="none", label_smoothing=0.1)(zd, t.to(DEV))
    nan = torch.isnan(m)
    assert bool(nan[0, 1, 2]) and int(nan.sum()) == 1
    m.backward(torch.ones_like(m))
    assert torch.isfinite(zd.grad).all() and float(zd.grad[0, :, 1, 2].abs().max()) == 0.0


@pytest.mark.parametrize("tdt,ii", [(torch.int64, -100), (torch.uint8, 255), (torch.int64, 2)])
def test_all_ignored_is_nan(tdt, ii):
    z = torch.randn(2, 4, 8, 8, device=DEV)
    t = torch.full((2, 8, 8), ii if ii >= 0 else -100, dtype=tdt, device=DEV)
    for kw in (dict(), dict(weight=torch.rand(4, device=DEV) + 0.5), dict(label_smoothing=0.2)):
        loss = b200seg.CrossEntropyLoss(ignore_index=ii, **kw)(z, t)
        assert torch.isnan(loss), kw
        ref = F.cross_entropy(z, t.long(), ignore_index=ii, **kw)
        assert torch.isnan(ref)
        assert float(b200seg.CrossEntropyLoss(ignore_index=ii, reduction="sum", **kw)(z, t)) == 0.0


@pytest.mark.parametrize("hw", [(64, 96), (63, 97)])
def test_explicit_default_arguments_run_the_default_kernel(hw, monkeypatch):
    """Spelled-out defaults take the original fused kernel, not the option kernels: the same gradient bit for bit, and the
    same loss up to the order of that kernel's f32 atomics (two calls of ``CrossEntropyLoss()`` differ the same way)."""
    from b200seg import ops
    H, W = hw
    z, t, _ = _case(4, 10, H, W, -100, torch.int64, seed=3)

    def fail(*a, **k):
        raise AssertionError("the option kernels ran for default arguments")

    outs = []
    for crit in (b200seg.CrossEntropyLoss(),
                 b200seg.CrossEntropyLoss(weight=None, ignore_index=-100, reduction="mean", label_smoothing=0.0)):
        monkeypatch.setattr(ops, "softmax_ce_ex", fail)
        zd = z.to(DEV).requires_grad_()
        loss = crit(zd, t.to(DEV))
        loss.backward()
        monkeypatch.undo()
        outs.append((loss.detach(), zd.grad))
    assert torch.equal(outs[0][1], outs[1][1])
    assert abs(float(outs[0][0]) - float(outs[1][0])) <= 1e-6 * abs(float(outs[0][0]))


@pytest.mark.parametrize("red", ["mean", "none"])
def test_cuda_graph_replay_equals_eager(red):
    B, C, H, W = 4, 10, 32, 64
    z, t, g = _case(B, C, H, W, 255, torch.uint8, seed=11)
    crit = b200seg.CrossEntropyLoss(weight=torch.rand(C, generator=g) + 0.5, ignore_index=255, reduction=red,
                                    label_smoothing=0.1).to(DEV)
    zs, ts = z.to(DEV).requires_grad_(), t.to(DEV)
    gout = torch.randn(B, H, W, generator=g).to(DEV)

    def step():
        zs.grad = None
        loss = crit(zs, ts)
        loss.backward(gout if red == "none" else None)
        return loss.detach(), zs.grad

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(s)
    eager_loss, eager_grad = (x.clone() for x in step())
    graph = torch.cuda.CUDAGraph()
    zs.grad = None
    with torch.cuda.graph(graph):
        gl, gg = step()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(gl, eager_loss)
    assert torch.equal(gg, eager_grad)


def test_f2_training_step_with_options_matches_torch_loss():
    """One MobileNetV2UNet training step from the trained F2 weights with weight + label_smoothing + uint8 targets with
    ignore_index=255, against the same step with torch.nn.CrossEntropyLoss on t.long(): both go through the same engine
    backward, so the parameter gradients differ only through d(logits)."""
    sd = f2_sd()
    x, t = O.road_scene_batch(2, 128, 256, seed=9300)
    g = torch.Generator().manual_seed(5)
    t8 = t.clone().to(torch.uint8)
    t8[torch.rand(t.shape, generator=g) < 0.1] = 255
    w = torch.rand(10, generator=g) + 0.5
    m = b200seg.MobileNetV2UNet(output_channels=10)
    full = dict(m.state_dict())
    full.update(expand_aliases(sd))
    m.load_state_dict(full, strict=True)
    m = m.to(DEV).train()
    xd = x.to(DEV)

    def grads(crit, target):
        m.zero_grad()
        loss = crit(m(xd), target)
        loss.backward()
        return float(loss), {k: p.grad.detach().double().clone() for k, p in m.named_parameters() if p.grad is not None}

    l_ours, g_ours = grads(b200seg.CrossEntropyLoss(weight=w, ignore_index=255, label_smoothing=0.1).to(DEV), t8.to(DEV))
    l_ref, g_ref = grads(torch.nn.CrossEntropyLoss(weight=w, ignore_index=255, label_smoothing=0.1).to(DEV), t8.long().to(DEV))
    assert abs(l_ours - l_ref) <= 1e-5 * abs(l_ref)
    assert g_ours.keys() == g_ref.keys() and len(g_ref) > 100
    top = max(float(b.abs().max()) for b in g_ref.values())
    compared, bad = 0, {}
    for k, b in g_ref.items():
        a = g_ours[k]
        if float(b.abs().max()) < 1e-5 * top:   # conv biases ahead of a train-mode BatchNorm: zero up to rounding noise
            continue
        compared += 1
        cos = float((a.flatten() @ b.flatten()) / (a.norm() * b.norm()))
        if cos < 0.99999 or _rel(a, b) > 1e-4:
            bad[k] = (cos, _rel(a, b), float(b.abs().max()))
    assert not bad, bad
    assert compared > 100
