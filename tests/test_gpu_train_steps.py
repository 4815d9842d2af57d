"""Every step of the training step, forward and backward, against float64 on the engine's own tensors.

End to end, a bf16 training step cannot be compared strictly with anything: one ReLU6 mask that flips in the forward moves a
deep gradient by tens of percent, in any implementation.  But given the tensors the forward saved, the backward is a linear
map, and each step of both passes can be checked locally.  ``train_path.run_backward(keep=...)`` records every tensor
gradient when it is complete and the dz each conv step feeds its gradient kernels.  Each step is then compared with a
float64 reference computed from the engine's own inputs to that step:

- forward: ``z`` against a float64 conv of the step's input with the operand the kernel reads (bf16-rounded master weights
  for the tensor-core dense convs, bf16 taps for the bf16 depthwise kernel, f32 otherwise); ``a`` against float64 BatchNorm
  with float64 batch statistics of the engine's ``z`` (+ activation, + residual); the running statistics, updated in place;
- backward: ``dz`` and the finalized d gamma / d beta against float64 autograd of BatchNorm + activation on the engine's
  ``z``, given the engine's incoming gradient; the weight and bias gradients in the arena against float64 autograd of the
  conv on the step's input and the kept ``dz``;
- wiring: every kept tensor gradient against the float64 sum, over all consumers of the tensor, of their adjoints applied to
  the engine's kept downstream gradients (conv data gradients with transposed weights and flipped taps, block shortcuts,
  both halves of upsample+concat, max pool, the output-layout step).

Bars: those of the per-kernel tests (test_gpu_train.py), which run the same kernels at the same operand precision, relative
to the reference tensor's maximum.  fp32: 3e-5 for activations and data gradients, 1e-4 for weight gradients, 2e-4 for the
BatchNorm backward; bf16: 8e-3, 1e-3 and 2e-2.  BatchNorm backward rule: the activation mask is recomputed from ``z`` in f32,
so an element that sits on a ReLU / ReLU6 boundary may flip its mask against the float64 reference; ``dz`` is therefore held
to the bar in the rms sense, and at most 1e-4 of its elements may exceed the bar in the max sense.  Per-channel sums over
pixels (d gamma, d beta, conv biases) may in addition be off by 1e-5 of the largest sum of the magnitudes of their terms:
several of them are analytically zero (a conv bias in front of a train-mode BatchNorm; d beta of a layer whose output only
reaches train-mode BatchNorms through 1x1 convs and shortcuts, such as features.11-17 of MobileNetV2), so their own maximum
is the rounding noise of the kernels' f32 partial sums (about 170 units of f32 rounding of that magnitude sum).
"""
import functools

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

import b200seg  # noqa: E402
from b200seg import ops, train_path  # noqa: E402
from b200seg._cabi import BF16, lib  # noqa: E402
from oracle import unet_oracle as O  # noqa: E402
from test_f2_fixture import _note  # noqa: E402  (the suite's parity-notes record)
from util import expand_aliases, f2_sd  # noqa: E402

DEV = "cuda"
BAR = {"fp32": dict(act=3e-5, wgrad=1e-4, bn=2e-4), "bf16": dict(act=8e-3, wgrad=1e-3, bn=2e-2)}
BN_OVER_FRACTION = 1e-4


def _nchw(t):
    return t.permute(0, 3, 1, 2).double()


@functools.lru_cache(maxsize=None)
def _f2():
    return expand_aliases(f2_sd())


def _model(arch):
    if arch == "mbv2":
        m = b200seg.MobileNetV2UNet(output_channels=10)
        full = dict(m.state_dict())
        full.update(_f2())
        m.load_state_dict(full, strict=True)
    else:
        m = b200seg.UNet(output_channels=10, base_filters=64)
        m.load_state_dict(O.synth_state_dict(O.unet_param_shapes(10, 64), seed=3), strict=True)
    return m.to(DEV).train()


def _inputs(arch, B, H, W, seed):
    if arch == "mbv2":
        x, t = O.road_scene_batch(B, H, W, seed=seed)
    else:
        x, t = O.synth_input(B, H, W, seed=seed), O.synth_target(B, H, W, seed=seed)
    return x.to(DEV).contiguous(), t.to(DEV).long()


def _dout(kind, out, t, seed):
    if kind == "ce":
        _, dl = ops.softmax_ce(out, t)          # the fused loss kernel's d(mean CE)/d(logits)
        return dl
    g = torch.Generator(device="cpu").manual_seed(seed)
    return torch.randn(out.shape, generator=g).to(DEV)


def _step(m, mode, dense_impl, x, t, dout_kind, ws=None):
    """One training step driven directly: forward, then backward with every gradient kept."""
    eng = m._get_engine()
    eng.precision, eng.dense_impl = mode, dense_impl
    running = {s.name: (s.bn.running_mean.clone(), s.bn.running_var.clone()) for s in eng.steps if s.bn is not None}
    with torch.no_grad():
        env, saved = train_path.run_forward(eng, x, mode)
        dout = _dout(dout_kind, env["out"], t, seed=5)
        ws = ws or train_path._workspace(eng)
        keep = {}
        train_path.run_backward(eng, env, saved, mode, dout, ws, keep=keep)
    torch.cuda.synchronize()
    return eng, env, saved, keep, ws, running


class Report:
    """Worst error of each quantity over the whole step; failures name the step, the quantity and the worst element."""

    def __init__(self, case, mode):
        self.case, self.bar, self.worst, self.fail = case, BAR["bf16" if mode == "bf16" else "fp32"], {}, []

    def _note(self, qty, step, err, bar):
        if qty not in self.worst or err > self.worst[qty][0]:
            self.worst[qty] = (err, step, bar)

    def _where(self, d, got, ref):
        i = int(d.flatten().argmax())
        idx = tuple(int(v) for v in torch.unravel_index(torch.tensor(i), d.shape))
        return f"worst at {idx}: got {float(got[idx]):.6g} ref {float(ref[idx]):.6g}"

    def max_rel(self, step, qty, got, ref, kind, note=None):
        got, ref = got.double(), ref.double()
        bar = self.bar[kind]
        d = (got - ref).abs()
        scale = float(ref.abs().max())
        err = float(d.max()) / max(scale, 1e-30)
        self._note(note or qty, step, err, bar)
        if not err < bar:
            self.fail.append(f"{step}: {qty} max error {err:.3e} of {scale:.3e} > {bar:g}; {self._where(d, got, ref)}")

    def sum_rel(self, step, qty, got, ref, kind, l1):
        """A per-channel sum over pixels: the bar of ``kind`` relative to the maximum, plus 1e-5 of the largest sum of the
        terms' magnitudes (``l1``), which bounds the f32 rounding of partial sums where the exact sum cancels."""
        got, ref = got.double(), ref.double()
        d = (got - ref).abs()
        allowed = self.bar[kind] * float(ref.abs().max()) + 1e-5 * l1
        err = float(d.max()) / max(allowed, 1e-30)
        self._note(qty + "_over_allowed", step, err, 1.0)
        if not err < 1.0:
            self.fail.append(f"{step}: {qty} max error {float(d.max()):.3e} > {allowed:.3e} allowed; {self._where(d, got, ref)}")

    def bn_dz(self, step, got, ref):
        """The BatchNorm-backward rule of the module docstring: rms bar, plus a bound on the elements over the max bar."""
        got, ref = got.double(), ref.double()
        bar = self.bar["bn"]
        d = (got - ref).abs()
        scale = max(float(ref.abs().max()), 1e-30)
        rms = float(d.pow(2).mean().sqrt()) / scale
        over = float((d > bar * scale).double().mean())
        self._note("dz_rms", step, rms, bar)
        self._note("dz_over_fraction", step, over, BN_OVER_FRACTION)
        self._note("dz_max", step, float(d.max()) / scale, None)
        if not (rms < bar and over <= BN_OVER_FRACTION):
            self.fail.append(f"{step}: dz rms error {rms:.3e} (bar {bar:g}), {over:.2e} of the elements over the max bar; "
                             f"{self._where(d, got, ref)}")

    def exact(self, step, qty, ok, msg):
        if not ok:
            self.fail.append(f"{step}: {qty}: {msg}")

    def finish(self, **paths):
        _note("train_steps_vs_f64", case=self.case, worst=self.worst, **paths)
        assert not self.fail, f"{len(self.fail)} failures in {self.case}:\n" + "\n".join(self.fail[:12])


def _is_tc(eng, mode):
    return mode == "bf16" and (eng.dense_impl or "tc") == "tc"


def _w_fwd(eng, s, mode):
    """The weights the forward kernel of step s reads, in float64 OIHW."""
    w = s.conv.weight.detach()
    if s.op != "stem" and _is_tc(eng, mode):           # conv_tc: bf16 packed weights; dwconv3x3_bf16w: bf16 taps
        return w.bfloat16().double()
    return w.double()


def _w_dgrad(eng, s, mode, saved):
    """The weights the data-gradient kernel of step s reads: the packed transposed operand for dense layers; for depthwise
    layers the flipped bf16 taps of the stride-1 kernel (bf16 tensor-core mode), else the f32 taps."""
    w = s.conv.weight.detach()
    if s.op == "dense" and _is_tc(eng, mode):
        return w.bfloat16().double()
    if s.op == "dw" and s.stride == 1 and "wbf" in saved[s.name]:
        return w.bfloat16().double()
    return w.double()


def _conv_args(s):
    k = s.conv.weight.shape[2]
    return dict(stride=s.stride, padding=k // 2, groups=s.conv.groups)


def _src64(s, env):
    return env[s.src].double() if s.op == "stem" else _nchw(env[s.src])      # the stem reads the NCHW input


def _act(y, act):
    return {ops.ACT_NONE: y, ops.ACT_RELU: F.relu(y), ops.ACT_RELU6: torch.clamp(y, 0, 6)}[act]


def _maxpool_adjoint(x64, dy64):
    """The gradient of 2x2 max pooling: each window's gradient goes to its first maximum in raster order."""
    B, C, H, W = x64.shape
    win = x64.reshape(B, C, H // 2, 2, W // 2, 2).permute(0, 1, 2, 4, 3, 5).reshape(B, C, H // 2, W // 2, 4)
    first = win.argmax(-1, keepdim=True)            # argmax returns the first of equal maxima
    g = torch.zeros_like(win).scatter_(-1, first, dy64.unsqueeze(-1))
    return g.reshape(B, C, H // 2, W // 2, 2, 2).permute(0, 1, 2, 4, 3, 5).reshape(B, C, H, W)


def _paths(eng, env, saved, mode):
    """Kernel chosen at the real shape of each step: conv_rs forward / data gradient, tap-row weight gradient, cluster or
    streamed BatchNorm in each direction."""
    tc = _is_tc(eng, mode)
    n_use = {}
    for s in eng.steps:
        for name in (s.src, s.res):
            if name:
                n_use[name] = n_use.get(name, 0) + 1
    paths = {}
    for s in eng.steps:
        if s.conv is None:
            continue
        tags = []
        B, H, W, cz = saved[s.name]["z"].shape
        cin = env[s.src].shape[1 if s.op == "stem" else -1]
        if s.op == "dense" and tc and s.taps == 9:
            rs_ok = ops.USE_CONV_RS and eng.tc_flags == 0
            if rs_ok and lib.b200seg_conv_rs_supported(H, W, cin, cz):
                tags.append("conv_rs")
            if rs_ok and lib.b200seg_conv_rs_supported(H, W, cz, cin) and (cin <= 32 or n_use[s.src] == 1):
                tags.append("conv_rs_dgrad")
            if W >= 128:
                tags.append("wgrad_taprow")
        if s.bn is not None and mode == "bf16" and ops.BN_CLUSTER:
            C = s.bn.weight.shape[0]
            tags.append("bn_cluster_fwd" if lib.b200seg_bn_cluster_supported(BF16, B * H * W, C) else "bn_streamed_fwd")
            tags.append("bn_cluster_bwd" if lib.b200seg_bn_cluster_bwd_supported(BF16, B * H * W, C) else "bn_streamed_bwd")
        paths[s.name] = tags
    return paths


def _check_step(m, mode, env, saved, keep, ws, running, rep):
    eng = m._get_engine()
    tc = _is_tc(eng, mode)
    steps = eng.steps
    by_dst = {s.dst: s for s in steps}
    views = ws.arena.views
    # ------------------------------------------------------------------ forward and parameter gradients, per step
    for s in steps:
        rec = saved[s.name]
        if s.op == "upcat":
            skip, xs = _nchw(env[s.res]), _nchw(env[s.src])
            ref = torch.cat([skip, F.interpolate(xs, scale_factor=2, mode="bilinear", align_corners=False)], 1)
            rep.max_rel(s.name, "fwd_upcat", _nchw(env[s.dst]), ref, "act")
            continue
        if s.op == "pool":
            rep.exact(s.name, "fwd_pool", torch.equal(_nchw(env[s.dst]), F.max_pool2d(_nchw(env[s.src]), 2)), "differs")
            continue
        if s.op in ("final", "to_nchw"):
            lg = _nchw(env[s.src])[:, :eng.out_ch]
            ref = F.interpolate(lg, scale_factor=2, mode="bilinear", align_corners=True) if s.op == "final" else lg
            rep.max_rel(s.name, "fwd_out", env[s.dst], ref, "act")
            continue
        cout = s.conv.weight.shape[0]
        x64 = _src64(s, env)
        b64 = s.conv.bias.detach().double() if s.conv.bias is not None else None
        z = rec["z"]
        zref = F.conv2d(x64, _w_fwd(eng, s, mode), b64, **_conv_args(s))
        rep.max_rel(s.name, "fwd_z", _nchw(z[..., :cout]), zref, "act")
        if z.shape[-1] > cout:                                   # Cout_pad columns of the logits: zero weights and bias
            rep.exact(s.name, "fwd_z_pad", float(z[..., cout:].abs().max()) == 0.0, "padded channels are not zero")
        z64 = _nchw(z[..., :cout])
        dz64 = _nchw(keep[("dz", s.name)][..., :cout])
        if s.bn is not None:
            bn = s.bn
            zz = z64.clone().requires_grad_(True)
            g64 = bn.weight.detach().double().requires_grad_(True)
            be64 = bn.bias.detach().double().requires_grad_(True)
            yb = F.batch_norm(zz, None, None, g64, be64, True, 0.0, bn.eps)
            yb.retain_grad()
            y = _act(yb, s.act)
            aref = y.detach() + (_nchw(env[s.res]) if s.res else 0.0)
            rep.max_rel(s.name, "fwd_a", _nchw(env[s.dst]), aref, "act")
            mean, var = z64.mean((0, 2, 3)), z64.var((0, 2, 3), unbiased=True)
            rm0, rv0 = running[s.name]
            mom = bn.momentum
            for qty, got, ref in (("running_mean", bn.running_mean, (1 - mom) * rm0.double() + mom * mean),
                                  ("running_var", bn.running_var, (1 - mom) * rv0.double() + mom * var)):
                d = (got.double() - ref).abs()
                rep.exact(s.name, qty, bool((d <= 1e-6 + 1e-5 * ref.abs()).all()),
                          f"worst channel {int(d.argmax())}: got {float(got[d.argmax()]):.7g} ref {float(ref[d.argmax()]):.7g}")
            y.backward(_nchw(keep[("d", s.dst)]))
            rep.bn_dz(s.name, dz64, zz.grad)
            xhat = (z64 - z64.mean((0, 2, 3), keepdim=True)) / (z64.var((0, 2, 3), unbiased=False, keepdim=True) + bn.eps).sqrt()
            rep.sum_rel(s.name, "dgamma", views[id(bn.weight)], g64.grad, "bn", float((yb.grad * xhat).abs().sum((0, 2, 3)).max()))
            rep.sum_rel(s.name, "dbeta", views[id(bn.bias)], be64.grad, "bn", float(yb.grad.abs().sum((0, 2, 3)).max()))
        else:
            rep.max_rel(s.name, "dz", keep[("dz", s.name)], keep[("d", s.dst)], "act")
        wref = torch.nn.grad.conv2d_weight(x64, s.conv.weight.shape, dz64, **_conv_args(s))
        rep.max_rel(s.name, "dweight", views[id(s.conv.weight)], wref, "wgrad")
        if s.conv.bias is not None:
            rep.sum_rel(s.name, "dbias", views[id(s.conv.bias)], dz64.sum((0, 2, 3)), "act", float(dz64.abs().sum((0, 2, 3)).max()))
    # ------------------------------------------------------------------ wiring: each tensor gradient = sum of its adjoints
    for (kind, name), got in keep.items():
        if kind != "d" or name == "out":
            continue
        shape = _nchw(env[name]).shape
        ref = torch.zeros(shape, device=DEV, dtype=torch.float64)
        for s in steps:
            if s.src == name and s.conv is not None:
                cout = s.conv.weight.shape[0]
                dz64 = _nchw(keep[("dz", s.name)][..., :cout])
                ref += torch.nn.grad.conv2d_input(shape, _w_dgrad(eng, s, mode, saved), dz64, **_conv_args(s))
            elif s.res == name and s.op == "dense":                      # block shortcut
                ref += _nchw(keep[("d", s.dst)])
            elif s.res == name and s.op == "upcat":                      # skip half of the concat
                ref += _nchw(keep[("d", s.dst)])[:, :shape[1]]
            elif s.src == name and s.op == "upcat":                      # upsampled half
                cs = env[s.res].shape[-1]
                xs = torch.zeros(shape, device=DEV, dtype=torch.float64, requires_grad=True)
                F.interpolate(xs, scale_factor=2, mode="bilinear", align_corners=False).backward(_nchw(keep[("d", s.dst)])[:, cs:])
                ref += xs.grad
            elif s.src == name and s.op == "pool":
                ref += _maxpool_adjoint(_nchw(env[name]), _nchw(keep[("d", s.dst)]))
            elif s.src == name and s.op in ("final", "to_nchw"):
                C = eng.out_ch
                dout = keep[("d", s.dst)].double()
                if s.op == "final":
                    lg = torch.zeros(shape[0], C, shape[2], shape[3], device=DEV, dtype=torch.float64, requires_grad=True)
                    F.interpolate(lg, scale_factor=2, mode="bilinear", align_corners=True).backward(dout)
                    dout = lg.grad
                ref[:, :C] += dout
        rep.max_rel(by_dst[name].name, f"d({name})", _nchw(got), ref, "act", note="dgrad_wiring")


CASES = {
    # name: (model, mode, dense_impl, (B, H, W), d(out))
    "mbv2-fp32": ("mbv2", "fp32", None, (2, 64, 128), "rand"),
    "mbv2-bf16-tc": ("mbv2", "bf16", None, (2, 64, 128), "rand"),
    "mbv2-bf16-tc-ce": ("mbv2", "bf16", None, (2, 64, 128), "ce"),
    "mbv2-bf16-simt": ("mbv2", "bf16", "simt", (2, 64, 128), "rand"),
    "mbv2-bf16-b8": ("mbv2", "bf16", None, (8, 128, 256), "ce"),
    "mbv2-bf16-256x512": ("mbv2", "bf16", None, (1, 256, 512), "rand"),
    "unet-bf16": ("unet", "bf16", None, (2, 64, 256), "ce"),
    "unet-fp32": ("unet", "fp32", None, (2, 64, 256), "rand"),
}


def _expect_paths(case, eng, paths):
    """What each case is there to reach; fails when a dispatch heuristic moves a kernel off the path a case covers."""
    ops_seen = {s.op for s in eng.steps}
    has = lambda tag: [n for n, t in paths.items() if tag in t]     # noqa: E731
    if case.startswith("mbv2"):
        assert {"stem", "dw", "dense", "upcat", "final"} <= ops_seen
        assert {s.stride for s in eng.steps if s.op == "dw"} == {1, 2}
        assert any(s.res for s in eng.steps if s.op == "dense")
    if case == "mbv2-bf16-b8":         # the F2 training batch: cluster BatchNorm at P = 1024 on the 576-channel layers
        assert "bn_cluster_bwd" in paths["backbone.features.12.conv.0"], paths
        assert "bn_cluster_fwd" in paths["backbone.features.13.conv.1"], paths
    if case == "mbv2-bf16-256x512":
        assert {"conv_rs", "conv_rs_dgrad", "wgrad_taprow"} <= set(paths["up4.conv.conv.0"]), paths
        assert "bn_streamed_bwd" in paths["backbone.features.2.conv.0"], paths
    if case == "unet-bf16":
        assert "pool" in ops_seen
        assert "wgrad_taprow" in paths["inc.conv.conv.3"], paths
        assert [n for n in has("bn_cluster_bwd") if eng.model.get_submodule(n).out_channels >= 128], paths
        assert not has("conv_rs") and not has("conv_rs_dgrad"), paths        # every 3x3 runs on conv_tc


@pytest.mark.parametrize("case", list(CASES))
def test_train_step_matches_float64_step_by_step(case):
    arch, mode, dense_impl, (B, H, W), dout_kind = CASES[case]
    m = _model(arch)
    x, t = _inputs(arch, B, H, W, seed=9200)
    eng, env, saved, keep, ws, running = _step(m, mode, dense_impl, x, t, dout_kind)
    paths = _paths(eng, env, saved, mode)
    _expect_paths(case, eng, paths)
    rep = Report(case, mode)
    _check_step(m, mode, env, saved, keep, ws, running, rep)
    rep.finish(paths={k: v for k, v in paths.items() if v})


def test_single_stream_backward_matches_two_streams(monkeypatch):
    """The weight-gradient side stream only reorders launches: with B200SEG_WGRAD_STREAM=0 (a fresh workspace) the arena
    gradients agree with the two-stream run to the rounding of the float atomics, 1e-5 of each tensor's maximum."""
    monkeypatch.delenv("B200SEG_WGRAD_STREAM", raising=False)
    m = _model("mbv2")
    x, t = _inputs("mbv2", 2, 64, 128, seed=9200)
    eng, env, saved, _, ws2, _ = _step(m, "bf16", None, x, t, "rand", ws=None)
    assert ws2.wg_stream is not None
    two = {k: v.clone() for k, v in ws2.arena.views.items()}
    monkeypatch.setenv("B200SEG_WGRAD_STREAM", "0")
    ws1 = train_path.TrainWorkspace(eng)
    assert ws1.wg_stream is None
    with torch.no_grad():
        train_path.run_backward(eng, env, saved, "bf16", _dout("rand", env["out"], t, seed=5), ws1)
    torch.cuda.synchronize()
    names = {id(p): n for n, p in m.named_parameters()}
    bad = []
    for k, a in two.items():
        d = float((ws1.arena.views[k] - a).abs().max())
        if d > 1e-5 * float(a.abs().max()):
            bad.append((names[k], d, float(a.abs().max())))
    assert not bad, bad
