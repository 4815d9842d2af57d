"""Training forward/backward of the drop-in models (model.train(): train.py:24,36,38).

One ``torch.autograd.Function`` spans the whole network: ``forward`` runs the fused step schedule with
train-mode BatchNorm (batch statistics, running-stat update, ``num_batches_tracked += 1``) and keeps, per
layer, the pre-BN conv output ``z``, the BN statistics and the activation output; ``backward`` walks the
schedule in reverse and returns one gradient per used parameter, so ``loss.backward()`` /
``optimizer.step()`` at the reference call sites work unchanged.  ``backbone.classifier`` is not on the path:
its ``.grad`` stays ``None`` exactly as in the reference (SURVEY finding 5).

Kernels: forward convs and the dense data gradients (same conv with transposed/flipped weights) go through
``conv_simt`` (f32) or ``conv_tc`` (bf16), dense weight gradients through ``conv_wgrad`` / ``conv_wgrad_tc``;
everything else is in csrc/train_ops.cu.  Gradient accumulation for tensors with two consumers (skip
connections, block inputs with a shortcut) rides on the conv kernels' ``+residual`` epilogue or the ``acc``
argument of the adjoint kernels -- there is no separate add pass.

Gradients: the backward kernels leave raw partial results (f64 slot sums, f32 accumulators in operand layout) in a
persistent staging buffer; one ``grad_finalize`` launch per bucket writes them, in parameter layout, into the flat
gradient arena (``dp.GradArena``) whose views ARE ``p.grad`` -- autograd never copies a parameter gradient.  With
``dp.attach`` each bucket's all-reduce is enqueued behind its finalize launch on a side stream and overlaps the rest
of backward, eagerly and inside the captured backward graph alike.

Steady state: after ``engine.graph_after`` steps with the same input shape, the forward and the backward are
each captured into a CUDA graph over static buffers (weight re-packing, gradient finalize and the collectives
included, so in-place optimizer updates are picked up); a step then costs two graph launches of host time instead of
~1600 kernel launches.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch

from . import ops
from .ops import ACT_NONE

TRACE = None      # set to a list to collect (phase, step name, start event, end event) per schedule step (eager only)


def _tick():
    if TRACE is None:
        return None
    e = torch.cuda.Event(enable_timing=True)
    e.record()
    return e


def _train_params(engine) -> List[torch.nn.Parameter]:
    ps = []
    for s in engine.steps:
        if s.conv is not None:
            ps.append(s.conv.weight)
            if s.conv.bias is not None:
                ps.append(s.conv.bias)
        if s.bn is not None:
            ps += [s.bn.weight, s.bn.bias]
    return ps


# ----------------------------------------------------------------------------------------------------
# weight repack: all layers in one launch (b200seg_pack_weights_multi) into persistent operand buffers
# ----------------------------------------------------------------------------------------------------
def _train_packs(engine, tc: bool):
    """Persistent packed-weight buffers of the training step + the device table that fills them.  Returns
    {step name: dict(wp=..., wk=..., wt=...)} after launching the repack for the CURRENT parameter values.
    (SURVEY 8f rank 1: before, every layer cost 3-6 tiny permute/cast/flip kernels per step, ~280 launches.)"""
    import ctypes
    from ._cabi import check, lib, ptr
    convs = [s for s in engine.steps if s.op in ("stem", "dw", "dense")]
    dev = convs[0].conv.weight.device
    key = (tc, dev, tuple(s.conv.weight.data_ptr() for s in convs))
    plan = getattr(engine, "_train_pack_plan", None)
    if plan is None or plan["key"] != key:
        chunk = int(lib.b200seg_pack_chunk())
        rows, views, ct, ci = [], {}, [], []
        n16 = n32 = 0
        metas = []
        dw16 = [s for s in convs if s.op == "dw"] if tc else []      # bf16 taps for the mixed-precision-FMA depthwise kernel
        for s in convs:
            w = s.conv.weight
            if not w.is_contiguous() or w.dtype != torch.float32:
                raise TypeError("training keeps contiguous fp32 master weights")
            cout, cin, k = w.shape[0], w.shape[1], w.shape[2]
            kk = k * k
            if s.op == "stem":
                kind, cp, nf, nd = 2, cout, kk * cin * cout, 0
            elif s.op == "dw":
                kind, cp, nf, nd = 3, cout, kk * cout, kk * cout
            else:
                kind = 0 if tc else 1
                cp = max(cout, s.pad_cout) if s.pad_cout else cout
                nf = nd = cp * kk * cin
            metas.append((s, kind, cout, cin, kk, cp, nf, nd))
            if s in dw16:
                metas.append((s, 4, cout, cin, kk, cp, nf, nd))
                n16 += 2 * ((nf + 7) // 8 * 8)
            if kind == 0:
                n16 += (nf + 7) // 8 * 8 + (nd + 7) // 8 * 8
            else:
                n32 += (nf + 3) // 4 * 4 + (nd + 3) // 4 * 4
        buf16 = torch.zeros(max(n16, 8), device=dev, dtype=torch.bfloat16)
        buf32 = torch.zeros(max(n32, 4), device=dev, dtype=torch.float32)
        o16 = o32 = 0
        for ti, (s, kind, cout, cin, kk, cp, nf, nd) in enumerate(metas):
            if kind in (0, 4):
                fwd = buf16[o16:o16 + nf]; o16 += (nf + 7) // 8 * 8
                dg = buf16[o16:o16 + nd]; o16 += (nd + 7) // 8 * 8
            else:
                fwd = buf32[o32:o32 + nf]; o32 += (nf + 3) // 4 * 4
                dg = buf32[o32:o32 + nd] if nd else None; o32 += (nd + 3) // 4 * 4
            if s.op == "stem":
                views[s.name] = dict(wp=fwd.view(s.conv.weight.shape[2], s.conv.weight.shape[3], cin, cout))
            elif s.op == "dw" and kind == 4:
                views[s.name].update(wb=fwd.view(kk, cout), wbf=dg.view(kk, cout))
            elif s.op == "dw":
                views[s.name] = dict(wp=fwd.view(kk, cout), wpf=dg.view(kk, cout))
            else:
                views[s.name] = dict(wk=fwd.view(cp, kk * cin), wt=dg.view(cin, kk * cp))
            # struct PackEntry {w, fwd, dgrad (8 bytes each); cout, cin, kk, cout_pad, kind, pad (4 bytes each)}
            rows += [s.conv.weight.data_ptr(), fwd.data_ptr(), dg.data_ptr() if dg is not None else 0,
                     (cin << 32) | cout, (cp << 32) | kk, kind]
            n = cp * cin * kk
            for c in range((n + chunk - 1) // chunk):
                ct.append(ti); ci.append(c)
        plan = dict(key=key, views=views, buf16=buf16, buf32=buf32, n=len(ct),
                    table=torch.tensor(rows, dtype=torch.int64, device=dev),
                    ct=torch.tensor(ct, dtype=torch.int32, device=dev), ci=torch.tensor(ci, dtype=torch.int32, device=dev))
        engine._train_pack_plan = plan
    check(lib.b200seg_pack_weights_multi(ptr(plan["table"]), ptr(plan["ct"]), ptr(plan["ci"]), plan["n"],
                                         torch.cuda.current_stream().cuda_stream), "pack_weights_multi")
    return plan["views"]


# ----------------------------------------------------------------------------------------------------
# gradient arena + staging + finalize tables (one per engine)
# ----------------------------------------------------------------------------------------------------
class TrainWorkspace:
    """Where the backward pass puts parameter gradients.

    ``arena``     dp.GradArena: flat fp32 buffer in backward order, bucketed; ``arena.views[id(p)]`` becomes ``p.grad``.
    ``stage``     {id(param): staging view the backward kernel of that parameter accumulates into}; BatchNorm's two
                  parameters share one f64 [NSLOT, 2, C] block (``stage[id(bn.weight)]``).
    ``finalize``  one ``b200seg_grad_finalize_multi`` launch per bucket: staging -> arena (parameter layout, * 1/world).
    ``wg_stream`` second CUDA stream for the weight-gradient kernels (``side``).  The data-gradient chain
                  dz -> dgrad -> BN backward -> dz of the layer before is the critical path of backward; the weight
                  gradient of a layer only needs dz and the saved input and nothing downstream needs it before the
                  bucket's finalize launch.  On the small deep layers neither kind of kernel fills 148 SMs (pixel-split
                  wgrad CTAs, 15-40 us each), so the two streams overlap; the fork/join events become graph edges
                  under capture.  ``B200SEG_WGRAD_STREAM=0`` keeps everything on one stream.
    """

    def __init__(self, engine):
        from . import dp
        from ._cabi import lib
        cfg = getattr(engine, "dp", None) or {}
        params = dp.used_parameters(engine.model)
        self.arena = dp.GradArena(params, cfg.get("group"), cfg.get("bucket_bytes", 8 << 20))
        dev = params[0].device
        NS = ops.NSLOT
        plan = []                     # (param, kind, which buffer, offset, numel, dims...)
        n64 = n32 = 0
        self._shape: Dict[int, tuple] = {}
        for s in engine.steps:
            if s.conv is None:
                continue
            w = s.conv.weight
            cout, cin, kk = w.shape[0], w.shape[1], w.shape[2] * w.shape[3]
            cp = max(cout, s.pad_cout) if s.pad_cout else cout
            if s.op == "stem":
                plan.append((w, 2, 32, n32, kk * cin * cout, cout, cin, kk, 0, 0)); self._shape[id(w)] = (w.shape[2], w.shape[3], cin, cout)
                n32 += (kk * cin * cout + 3) // 4 * 4
            elif s.op == "dw":
                plan.append((w, 3, 64, n64, NS * kk * cout, cout, 1, kk, NS, kk * cout)); self._shape[id(w)] = (NS, kk, cout)
                n64 += NS * kk * cout
            else:
                plan.append((w, 1, 32, n32, cp * kk * cin, cout, cin, kk, 0, 0)); self._shape[id(w)] = (cp, kk * cin)
                n32 += (cp * kk * cin + 3) // 4 * 4
            if s.conv.bias is not None:
                b = s.conv.bias
                plan.append((b, 0, 64, n64, NS * cp, cout, 0, 0, NS, cp)); self._shape[id(b)] = (NS, cp)
                n64 += NS * cp
            if s.bn is not None:
                C = s.bn.weight.shape[0]
                # [NSLOT][2][C]: row 0 = sum g (d beta), row 1 = sum g*xhat (d gamma)
                plan.append((s.bn.bias, 0, 64, n64, NS * 2 * C, C, 0, 0, NS, 2 * C)); self._shape[id(s.bn.bias)] = (NS, 2, C)
                plan.append((s.bn.weight, 0, 64, n64 + C, 0, C, 0, 0, NS, 2 * C))
                n64 += NS * 2 * C
        self.s64 = torch.zeros(max(n64, 1), device=dev, dtype=torch.float64)
        self.s32 = torch.zeros(max(n32, 1), device=dev, dtype=torch.float32)
        self.stage: Dict[int, torch.Tensor] = {}
        src_ptr: Dict[int, int] = {}
        meta: Dict[int, tuple] = {}
        for (p, kind, buf, off, numel, cout, cin, kk, nslot, sstride) in plan:
            base = self.s64 if buf == 64 else self.s32
            if numel:
                self.stage[id(p)] = base[off:off + numel].view(self._shape[id(p)])
            src_ptr[id(p)] = base.data_ptr() + off * base.element_size()
            meta[id(p)] = (kind, cout, cin, kk, nslot, sstride)
        for s in engine.steps:          # BatchNorm: both parameters are staged in the block registered under bn.bias
            if s.bn is not None:
                self.stage[id(s.bn.weight)] = self.stage[id(s.bn.bias)]
        # finalize table (arena order) + per-bucket chunk lists
        import struct
        chunk = int(lib.b200seg_grad_chunk())
        scale_bits = struct.unpack("<I", struct.pack("<f", 1.0 / self.arena.world))[0]
        rows = []
        index = {}
        for ti, p in enumerate(self.arena.params):
            kind, cout, cin, kk, nslot, sstride = meta[id(p)]
            index[id(p)] = ti
            rows += [self.arena.views[id(p)].data_ptr(), src_ptr[id(p)], p.numel(), sstride,
                     (cout << 32) | kind, (kk << 32) | cin, nslot, scale_bits]
        self.table = torch.tensor(rows, dtype=torch.int64, device=dev)
        self.bucket_chunks = []
        for b in self.arena.buckets:
            ct, ci = [], []
            for p in b["params"]:
                for c in range((p.numel() + chunk - 1) // chunk):
                    ct.append(index[id(p)]); ci.append(c)
            self.bucket_chunks.append((torch.tensor(ct, dtype=torch.int32, device=dev),
                                       torch.tensor(ci, dtype=torch.int32, device=dev), len(ct)))
        self.pending: List[int] = []
        import os
        self.wg_stream = (torch.cuda.Stream(device=dev)
                          if dev.type == "cuda" and os.environ.get("B200SEG_WGRAD_STREAM", "1") != "0" else None)
        self._wg_forked = False
        self._wg_keep: list = []      # tensors the side stream still reads (must outlive the main stream's references)

    def begin_backward(self) -> None:
        self.s64.zero_()
        self.s32.zero_()
        self.pending = [len(b["params"]) for b in self.arena.buckets]

    def side(self, fn, *reads) -> None:
        """Run ``fn`` (weight-gradient launches reading ``reads``) behind everything enqueued so far, off the critical path."""
        if self.wg_stream is None:
            fn()
            return
        self.wg_stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.wg_stream):
            fn()
        self._wg_keep.extend(reads)
        self._wg_forked = True

    def join_side(self) -> None:
        if self._wg_forked:
            torch.cuda.current_stream().wait_stream(self.wg_stream)
            self._wg_forked = False
        self._wg_keep.clear()

    def done(self, *params) -> None:
        """The staging of these parameters is complete (their kernels are enqueued).  When a bucket fills: finalize it into
        the arena and start its all-reduce behind that launch."""
        from ._cabi import check, lib, ptr
        for p in params:
            bi = self.arena.bucket_of[id(p)]
            self.pending[bi] -= 1
            if self.pending[bi] == 0:
                self.join_side()                 # the bucket's weight gradients are complete
                ct, ci, n = self.bucket_chunks[bi]
                check(lib.b200seg_grad_finalize_multi(ptr(self.table), ptr(ct), ptr(ci), n,
                                                      torch.cuda.current_stream().cuda_stream), "grad_finalize_multi")
                self.arena.reduce_bucket(bi)

    def end_backward(self) -> None:
        if any(self.pending):
            raise RuntimeError("gradient bucket incomplete: a parameter on the path produced no gradient")
        self.join_side()
        self.arena.join()


def _workspace(engine) -> TrainWorkspace:
    ws = getattr(engine, "_train_ws", None)
    key = tuple(p.data_ptr() for p in _train_params(engine))
    if ws is None or ws.key != key:
        ws = TrainWorkspace(engine)
        ws.key = key
        engine._train_ws = ws
    return ws


# ----------------------------------------------------------------------------------------------------
# the two passes as plain functions over tensors (no autograd): used eagerly and under graph capture
# ----------------------------------------------------------------------------------------------------
def _out_step(engine):
    """The last schedule step when it only produces the public output layout (final upsample / NHWC->NCHW), else None."""
    last = engine.steps[-1]
    return last if last.op in ("final", "to_nchw") else None


def run_out_step(engine, s, env):
    """Forward of the output-layout step into a FRESH tensor."""
    if s.op == "final":
        return ops.upsample2x_ac_nchw(env[s.src], engine.out_ch, torch.float32)
    return ops.nhwc_to_nchw(env[s.src], engine.out_ch, torch.float32)


def run_out_step_bwd(engine, s, env, dout, sdt, out=None):
    """Backward of the output-layout step: reads the caller's d(out) directly."""
    if s.op == "final":
        return ops.final_bwd(dout, sdt, env[s.src].shape[-1], out=out)
    return ops.nchw_to_nhwc_pad(dout, env[s.src].shape[-1], sdt, out=out)


def run_forward(engine, x: torch.Tensor, mode: str, skip_out_step: bool = False):
    sdt = torch.bfloat16 if mode == "bf16" else torch.float32
    tc = mode == "bf16" and (engine.dense_impl or "tc") == "tc"
    env: Dict[str, torch.Tensor] = {"x": x}
    saved: Dict[str, dict] = {}
    ops.zero_pool.reset()
    ops.zero_pool32.reset()
    packs = _train_packs(engine, tc)       # every layer's operand layouts from the current fp32 weights, one launch
    counters = []                          # BatchNorm.num_batches_tracked, bumped with one fused launch at the end
    out_step = _out_step(engine) if skip_out_step else None
    for s in engine.steps:
        rec: dict = {}
        _e0 = _tick()
        if s is out_step:                      # launched by the caller outside the captured graph (fresh output tensor)
            saved[s.name] = rec
            continue
        if s.op in ("stem", "dw", "dense"):
            cout = s.conv.weight.shape[0]
            bias = s.conv.bias.detach().float() if s.conv.bias is not None else None
            src = env[s.src]
            pk = packs[s.name]
            if s.op == "stem":
                rec["wp"] = pk["wp"]
                z = ops.conv3x3_smallcin(src, rec["wp"], bias, s.stride, ACT_NONE, sdt)
            elif s.op == "dw":
                rec["wp"], rec["wpf"] = pk["wp"], pk["wpf"]
                if "wb" in pk:          # bf16 activations: mixed-precision-FMA kernel with bf16 taps
                    rec["wbf"] = pk["wbf"]
                    z = ops.dwconv3x3_bf16w(src, pk["wb"], bias, s.stride, ACT_NONE)
                else:
                    z = ops.dwconv3x3(src, rec["wp"], bias, s.stride, ACT_NONE)
            else:
                if s.pad_cout and cout < s.pad_cout and bias is not None:
                    bias = torch.cat([bias, bias.new_zeros(s.pad_cout - cout)], 0)
                rec["wk"], rec["wt"] = pk["wk"], pk["wt"]     # [Cout_pad, taps*Cin] and its transposed/tap-flipped twin
                if tc:
                    z = ops.conv_tc(src, rec["wk"], bias, s.taps, ACT_NONE, None, flags=engine.tc_flags)
                else:
                    z = ops.conv_simt(src, rec["wk"], bias, s.taps, ACT_NONE, None)
            rec["z"] = z
            if s.bn is not None:
                res = env[s.res] if (s.op == "dense" and s.res) else None
                a, sv = ops.bn_train_forward(z, s.bn.weight.detach().float(), s.bn.bias.detach().float(),
                                             s.bn.running_mean, s.bn.running_var, s.bn.eps,
                                             s.bn.momentum, s.act, res)
                counters.append(s.bn.num_batches_tracked)
                rec["sv"] = sv
                env[s.dst] = a
            else:
                env[s.dst] = z
        elif s.op == "upcat":
            env[s.dst] = ops.upsample2x_concat(env[s.res], env[s.src])
        elif s.op == "pool":
            env[s.dst] = ops.maxpool2x2(env[s.src])
        elif s.op in ("final", "to_nchw"):
            env[s.dst] = run_out_step(engine, s, env)
        else:  # pragma: no cover
            raise AssertionError(s.op)
        saved[s.name] = rec
        if _e0 is not None:
            TRACE.append(("fwd", s.name, _e0, _tick()))
    if counters:
        torch._foreach_add_(counters, 1)
    return env, saved


def run_backward(engine, env, saved, mode: str, dout, ws: TrainWorkspace, g_src=None, keep: Optional[dict] = None) -> None:
    """Walk the schedule in reverse.  Parameter gradients are accumulated in ``ws`` staging; as soon as the last
    parameter of a gradient bucket is staged the bucket is finalized into the arena and (data parallel) its all-reduce
    starts on the side stream while the walk continues.

    ``keep`` (dict, as in ``engine.forward_eval``) receives a clone of every tensor gradient at the moment it is complete,
    under ("d", tensor name), and of the dz each conv step feeds its weight- and data-gradient kernels, under
    ("dz", step name).  Clones, because a gradient is handed on unchanged as the shortcut gradient of a block input."""
    sdt = torch.bfloat16 if mode == "bf16" else torch.float32
    tc = mode == "bf16" and (engine.dense_impl or "tc") == "tc"
    # g_src: the gradient of the output-layout step's INPUT, already computed by the caller outside the captured graph
    out_step = _out_step(engine) if g_src is not None else None
    g: Dict[str, torch.Tensor] = {"out": dout} if out_step is None else {out_step.src: g_src}

    def pop(name):
        t = g.pop(name)
        if keep is not None:
            keep[("d", name)] = t.clone()
        return t

    ops.zero_pool.reset()
    ops.zero_pool32.reset()
    ws.begin_backward()
    for s in reversed(engine.steps):
        rec = saved[s.name]
        _e0 = _tick()
        if s is out_step:
            continue
        if s.op in ("final", "to_nchw"):
            g[s.src] = run_out_step_bwd(engine, s, env, pop(s.dst), sdt)
        elif s.op == "upcat":
            dcat = pop(s.dst)
            cs = env[s.res].shape[-1]
            dskip, dx = ops.upcat_bwd(dcat, cs, g.get(s.res))
            g[s.res] = dskip
            assert s.src not in g
            g[s.src] = dx
        elif s.op == "pool":
            g[s.src] = ops.maxpool_bwd(env[s.src], pop(s.dst), g.get(s.src))
        else:
            da = pop(s.dst)
            z = rec["z"]
            if s.bn is not None:
                if s.op == "dense" and s.res:           # shortcut: the same gradient flows to the block input
                    assert s.res not in g
                    g[s.res] = da
                dz, _, _ = ops.bn_train_backward(da, z, rec["sv"], s.act, red=ws.stage[id(s.bn.weight)])
                ws.done(s.bn.weight, s.bn.bias)
            else:
                dz = da                                   # conv + bias only (the last 1x1 of outconv)
            if keep is not None:
                keep[("dz", s.name)] = dz.clone()
            w = s.conv.weight
            if s.conv.bias is not None:
                ws.side(lambda: ops.colsum(dz, acc=ws.stage[id(s.conv.bias)]), dz)
                ws.done(s.conv.bias)
            src = env[s.src]
            if s.op == "stem":
                ws.side(lambda: ops.smallcin_wgrad(src, dz, s.stride, dw=ws.stage[id(w)]), src, dz)   # [3,3,Cin,Cout]
                ws.done(w)
            elif s.op == "dw":
                ws.side(lambda: ops.dw_wgrad(src, dz, s.stride, acc=ws.stage[id(w)]), src, dz)        # f64 slots [NSLOT,9,C]
                ws.done(w)
                if s.stride == 1 and g.get(s.src) is None:
                    # stride 1: the data gradient IS the forward depthwise conv of dz with the taps flipped -> the
                    # register-blocked forward kernel (2.5x faster than the generic gather kernel)
                    if "wbf" in rec:
                        g[s.src] = ops.dwconv3x3_bf16w(dz, rec["wbf"], None, 1, ACT_NONE)
                    else:
                        g[s.src] = ops.dwconv3x3(dz, rec["wpf"], None, 1, ACT_NONE)
                else:
                    g[s.src] = ops.dw_dgrad(dz, rec["wp"], tuple(src.shape), s.stride, g.get(s.src))
            else:
                if tc:
                    ws.side(lambda: ops.conv_wgrad_tc(src, dz, s.taps, dw=ws.stage[id(w)]), src, dz)  # [Cout_pad, taps*Cin]
                else:
                    ws.side(lambda: ops.conv_wgrad(src, dz, s.taps, dw=ws.stage[id(w)]), src, dz)
                ws.done(w)
                # dgrad = the same conv with W transposed (and the 3x3 taps flipped): packed with the forward operand
                wt = rec["wt"]                                          # [Cin, taps*Cout_pad]
                if tc:
                    g[s.src] = ops.conv_tc(dz, wt, None, s.taps, ACT_NONE, g.get(s.src), flags=engine.tc_flags)
                else:
                    g[s.src] = ops.conv_simt(dz, wt, None, s.taps, ACT_NONE, g.get(s.src))
        if _e0 is not None:
            TRACE.append(("bwd", s.name, _e0, _tick()))
    ws.end_backward()


# ----------------------------------------------------------------------------------------------------
# CUDA-graph replay of the two passes
# ----------------------------------------------------------------------------------------------------
class _StepGraph:
    """Forward and backward graphs of one (input shape, dtype, mode), sharing one memory pool."""

    def __init__(self, engine, x: torch.Tensor, mode: str):
        self.x = torch.empty_like(x)
        self.x.copy_(x)
        # torch.cuda.graph() does not run the captured work, but BatchNorm's num_batches_tracked bump is captured
        # like any other kernel, so nothing is double counted.
        # build the persistent repack plan and the gradient workspace (allocations, table uploads) OUTSIDE the capture
        _train_packs(engine, mode == "bf16" and (engine.dense_impl or "tc") == "tc")
        ws = _workspace(engine)
        torch.cuda.synchronize()
        from ._cabi import LAUNCHES
        n0 = LAUNCHES[0]
        self.fwd = torch.cuda.CUDAGraph()
        # The output-layout step (final upsample) and its adjoint stay OUTSIDE the graphs: the forward one writes a fresh
        # result tensor, the backward one reads the caller's d(out) -- no 168 MB clone / copy_ around the replays.
        self.out_step = _out_step(engine)
        with torch.no_grad(), torch.cuda.graph(self.fwd):
            self.env, self.saved = run_forward(engine, self.x, mode, skip_out_step=True)
        sdt = torch.bfloat16 if mode == "bf16" else torch.float32
        if self.out_step is not None:
            self.out = None
            self.dout = None
            self.g_src = torch.zeros_like(self.env[self.out_step.src], dtype=sdt)
        else:
            self.out = self.env["out"]
            self.dout = torch.zeros_like(self.out)
            self.g_src = None
        self.bwd = torch.cuda.CUDAGraph()
        # the per-bucket all-reduces (data parallel) are captured on the arena's side stream: fork/join events become
        # graph edges, so every replay overlaps them with the rest of backward
        with torch.no_grad(), torch.cuda.graph(self.bwd, pool=self.fwd.pool()):
            run_backward(engine, self.env, self.saved, mode, self.dout, ws, g_src=self.g_src)
        self.n_launches = LAUNCHES[0] - n0     # hand-written kernels inside the two graphs (ATen fills/copies not counted)
        self.pending = False      # a forward has been replayed whose backward has not run yet


def _detach_accumulated(params, ws) -> None:
    """Gradient accumulation: a ``p.grad`` that still aliases the arena (the caller did not zero_grad to None) would be
    overwritten by this backward; give it storage of its own first."""
    for p in params:
        g = p.grad
        if g is not None and g.data_ptr() == ws.arena.views[id(p)].data_ptr():
            p.grad = g.clone()


def _assign_grads(params, ws) -> None:
    for p in params:
        v = ws.arena.views[id(p)]
        if p.grad is None:
            p.grad = v if p.dtype == torch.float32 else v.to(p.dtype)
        else:
            p.grad.add_(v)


class _TrainFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, engine, allow_graph, x, *params):
        mode = engine._mode(x)
        x = x.contiguous()
        ctx.engine, ctx.mode, ctx.graph = engine, mode, None
        ops.bump_mutation_epoch()            # BatchNorm running stats / counters change below, also under graph replay
        sg = _graph_for(engine, x, mode) if allow_graph else None
        if sg is not None:
            sg.x.copy_(x)
            sg.fwd.replay()
            sg.pending = True
            ctx.graph = sg
            out = run_out_step(engine, sg.out_step, sg.env) if sg.out_step is not None else sg.out.clone()
        else:
            with torch.no_grad():
                ctx.env, ctx.saved = run_forward(engine, x, mode)
            out = ctx.env["out"]
        return out.to(x.dtype) if x.dtype != torch.float32 else out

    @staticmethod
    def backward(ctx, dout):
        engine = ctx.engine
        params = _train_params(engine)
        none = (None, None, None, *[None] * len(params))       # parameter gradients are assigned to p.grad directly
        with torch.cuda.device(dout.device):
            ws = _workspace(engine)
            _detach_accumulated(params, ws)
            sg = ctx.graph
            if sg is not None:
                if sg.out_step is not None:
                    sdt = torch.bfloat16 if ctx.mode == "bf16" else torch.float32
                    run_out_step_bwd(engine, sg.out_step, sg.env, dout.float().contiguous(), sdt, out=sg.g_src)
                else:
                    sg.dout.copy_(dout)
                sg.bwd.replay()
                sg.pending = False
                ctx.graph = None             # the loss tensor's autograd node must not keep the captured graphs alive
            else:
                with torch.no_grad():
                    run_backward(engine, ctx.env, ctx.saved, ctx.mode, dout.float().contiguous(), ws)
                ctx.env = ctx.saved = None
            _assign_grads(params, ws)
        return none


def _graph_for(engine, x, mode) -> Optional[_StepGraph]:
    """The step graph to replay for this call, or None (eager): graphs need grad mode, no tracing, a warmed-up
    shape, and no forward still waiting for its backward (two forwards would share the static buffers)."""
    if not engine.use_graphs or TRACE is not None or torch.cuda.is_current_stream_capturing():
        return None
    # the captured graphs hold raw pointers of every parameter and BatchNorm buffer: a graph is only valid for them
    key = ("train", tuple(x.shape), x.dtype, mode, engine.dense_impl, engine.tc_flags, x.device, engine._ptr_ident(),
           id(getattr(engine, "dp", None)))
    ent = engine._graphs.get(key)
    if ent is None:
        if len(engine._graphs) >= 3:
            engine._graphs.clear()
        ent = engine._graphs[key] = {"seen": 0, "graph": None}
    ent["seen"] += 1
    if ent["graph"] is None and ent["seen"] > engine.graph_after:
        ent["graph"] = _StepGraph(engine, x, mode)
    sg = ent["graph"]
    if sg is None or sg.pending:
        return None
    return sg


def _check_bn_modes(engine) -> None:
    """The fused training path implements nn.BatchNorm2d's defaults as the reference uses them; anything else must fail
    loudly instead of silently training differently."""
    for s in engine.steps:
        bn = s.bn
        if bn is None:
            continue
        if not bn.training:
            raise NotImplementedError(f"{s.name}: per-module bn.eval() inside model.train() is not supported")
        if bn.momentum is None or not bn.track_running_stats or not bn.affine:
            raise NotImplementedError(f"{s.name}: BatchNorm2d(momentum=None / track_running_stats=False / affine=False) "
                                      "is not supported by the fused training path")


def forward_train(engine, x: torch.Tensor) -> torch.Tensor:
    params = _train_params(engine)
    engine._check_input(x)
    _check_bn_modes(engine)
    if params[0].dtype != torch.float32:
        raise TypeError("training keeps fp32 master weights: use model.float() and engine.precision='bf16' "
                        "(or torch.autocast) for bf16 activations")
    if not torch.is_grad_enabled():
        # model.train() under no_grad (e.g. BN calibration): forward only, still updates running stats
        return _TrainFn.apply(engine, False, x, *[p.detach() for p in params])
    return _TrainFn.apply(engine, True, x, *params)
