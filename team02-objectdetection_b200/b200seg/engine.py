"""Execution engine behind ``MobileNetV2UNet.forward`` / ``UNet.forward``.

The nn.Module tree (b200seg.unet) only *holds* parameters.  This module turns it into a static
list of fused steps -- conv(+BN)(+act)(+residual), depthwise conv(+BN+ReLU6), upsample+concat,
final upsample -- packs the weights once per parameter version (BN folded in fp32, K-major bf16 for
the tensor-core path) and launches the sm_100a kernels through the C ABI.

Data layout in HBM: activations NHWC (channels innermost, 16-byte aligned rows) in the storage
dtype (bf16 on the tensor-core path, f32 on the exact path); the public input/output stay NCHW as
in the reference (unet.py:32-51): the stem kernel reads NCHW directly and the final upsample kernel
writes NCHW directly, so no layout-conversion pass exists.

Precision modes
  "bf16": bf16 activations + tcgen05 convs (fp32 accumulate).  Chosen when the module is .bfloat16(),
          under torch.autocast(bfloat16), or after ``model.set_precision("bf16")``.
  "fp32": f32 activations + FP32-pipe convs: the 1e-4-relative configuration (BASELINE config 1).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, List, Optional

import torch
import torch.nn as nn

from . import ops
from .ops import ACT_NONE, ACT_RELU, ACT_RELU6


@dataclass
class Step:
    op: str                      # stem | dw | dense | upcat | pool | final | to_nchw
    name: str                    # module path (debug / profiling labels)
    src: str
    dst: str
    conv: Optional[nn.Conv2d] = None
    bn: Optional[nn.BatchNorm2d] = None
    act: int = ACT_NONE
    stride: int = 1
    taps: int = 1
    res: Optional[str] = None    # residual source (dense) / skip source (upcat)
    pad_cout: int = 0            # pad output channels (logits 10 -> 16)
    parts: Optional[tuple] = None   # op == "mbconv": the (expand, depthwise, project) steps it replaces


def _double_conv_steps(prefix: str, dc, src: str, dst: str) -> List[Step]:
    seq = dc.conv
    return [Step("dense", f"{prefix}.conv.0", src, dst + ".a", seq[0], seq[1], ACT_RELU, taps=9),
            Step("dense", f"{prefix}.conv.3", dst + ".a", dst, seq[3], seq[4], ACT_RELU, taps=9)]


def _outconv_steps(prefix: str, oc, src: str, dst: str) -> List[Step]:
    seq = oc.conv
    ncls = seq[3].weight.shape[0]            # logits are stored NHWC with the class axis padded to a multiple of 16
    return [Step("dense", f"{prefix}.conv.0", src, dst + ".a", seq[0], seq[1], ACT_RELU, taps=1),
            Step("dense", f"{prefix}.conv.3", dst + ".a", dst, seq[3], None, ACT_NONE, taps=1, pad_cout=(ncls + 15) // 16 * 16)]


def build_steps_mbv2unet(model) -> List[Step]:
    """Static schedule of MobileNetV2UNet.forward (unet.py:32-51)."""
    f = model.backbone.features
    st: List[Step] = [Step("stem", "backbone.features.0", "x", "f0", f[0][0], f[0][1], ACT_RELU6, stride=2, taps=9)]
    for i in range(1, 18):
        blk, seq, p = f[i], f[i].conv, f"backbone.features.{i}"
        src, j = f"f{i - 1}", 0
        if blk.expand_ratio != 1:
            st.append(Step("dense", f"{p}.conv.0", src, f"f{i}.e", seq[0][0], seq[0][1], ACT_RELU6))
            src, j = f"f{i}.e", 1
        st.append(Step("dw", f"{p}.conv.{j}", src, f"f{i}.d", seq[j][0], seq[j][1], ACT_RELU6, stride=blk.stride, taps=9))
        st.append(Step("dense", f"{p}.conv.{j + 1}", f"f{i}.d", f"f{i}", seq[j + 1], seq[j + 2], ACT_NONE,
                       res=f"f{i - 1}" if blk.use_res_connect else None))
    st.append(Step("dense", "backbone.features.18", "f17", "f18", f[18][0], f[18][1], ACT_RELU6))
    cur = "f18"
    for k, skip in ((1, "f10"), (2, "f6"), (3, "f3"), (4, "f1")):       # unet.py:41-44
        st.append(Step("upcat", f"up{k}.up", cur, f"up{k}.cat", res=skip))
        st += _double_conv_steps(f"up{k}.conv", getattr(model, f"up{k}").conv, f"up{k}.cat", f"up{k}")
        cur = f"up{k}"
    st += _outconv_steps("outc", model.outc, cur, "logits")
    st.append(Step("final", "final_upsample", "logits", "out"))
    return st


def build_steps_unet(model) -> List[Step]:
    """Static schedule of UNet.forward (unet.py:137-147)."""
    seq = model.inc.conv.conv
    st: List[Step] = [Step("stem", "inc.conv.conv.0", "x", "x1.a", seq[0], seq[1], ACT_RELU, stride=1, taps=9),
                      Step("dense", "inc.conv.conv.3", "x1.a", "x1", seq[3], seq[4], ACT_RELU, taps=9)]
    for k in (1, 2, 3):
        st.append(Step("pool", f"down{k}.mpconv.0", f"x{k}", f"x{k}.p"))
        st += _double_conv_steps(f"down{k}.mpconv.1", getattr(model, f"down{k}").mpconv[1], f"x{k}.p", f"x{k + 1}")
    cur = "x4"
    for k, skip in ((1, "x3"), (2, "x2"), (3, "x1")):
        st.append(Step("upcat", f"up{k}.up", cur, f"up{k}.cat", res=skip))
        st += _double_conv_steps(f"up{k}.conv", getattr(model, f"up{k}").conv, f"up{k}.cat", f"up{k}")
        cur = f"up{k}"
    st += _outconv_steps("sem_out", model.sem_out, cur, "logits")
    st.append(Step("to_nchw", "output", "logits", "out"))
    return st


class Engine:
    def __init__(self, model, arch: str):
        self.model = model
        self.arch = arch
        self.steps = build_steps_mbv2unet(model) if arch == "mbv2unet" else build_steps_unet(model)
        self.precision: Optional[str] = None       # None = derive from module dtype / autocast
        self.dense_impl: Optional[str] = None       # None = "tc" for bf16, "simt" for fp32 (tests may force)
        self.dw_impl: Optional[str] = None          # None = per-layer choice; "tc" / "simt" force one kernel
        self.mbconv_impl: Optional[str] = None      # None = per-block choice; "fused" / "unfused" force (eval bf16 only)
        self.tail_impl: Optional[str] = None        # None = fused outconv + final upsample (+argmax) when it applies; "unfused"
        self.head_impl: Optional[str] = None        # None = fused features.0 + features.1 (stem_mb1) when it applies; "unfused"
        self.mbconv_flags = 0
        self._eval_sched: Dict[tuple, List[Step]] = {}
        self.tc_flags = 0
        self._packed: Dict[str, dict] = {}
        self._packed_key = None
        self._graphs: Dict[tuple, dict] = {}
        self.use_graphs = True            # replay the steady-state forward from a CUDA graph
        self.graph_after = 2              # eager calls per (shape, weights) before capturing
        self.divisor = 32 if arch == "mbv2unet" else 8
        self.out_ch = model.output_channels
        self.dp = None                    # data parallel: set by b200seg.dp.attach() (group, bucket size)
        self._train_ws = None             # gradient arena + staging (train_path.TrainWorkspace)

    # ------------------------------------------------------------------ weights
    def _version_items(self):
        """(owning dict, name, tensor) of every parameter and buffer, built once: walking the module tree through
        ``model.parameters()`` costs ~1 ms of host time per forward (379 tensors), more than half of what the host spends on a
        whole 1.9 ms inference step."""
        items = []
        for mod in self.model.modules():
            for d in (mod._parameters, mod._buffers):
                for name, t in d.items():
                    if t is not None:
                        items.append((d, name, t))
        return items

    def _ptr_ident(self) -> int:
        """Hash of the storage addresses of every parameter and buffer (what a captured graph holds raw pointers to)."""
        items = getattr(self, "_ver_items", None)
        if items is None or any(d.get(name) is not t for d, name, t in items):
            items = self._ver_items = self._version_items()
        return hash(tuple(t.data_ptr() for _, _, t in items))

    def _version_key(self, mode: str):
        items = getattr(self, "_ver_items", None)
        if items is None:
            items = self._ver_items = self._version_items()
        v = 0
        for d, name, t in items:
            if d.get(name) is not t:          # a parameter/buffer object was replaced (load_state_dict(assign=True), p = nn.Parameter(..))
                items = self._ver_items = self._version_items()
                v = -1
                break
            v += t._version
        if v < 0:
            v = 0
            for d, name, t in items:
                v += t._version
            # id(items) in the key forces a re-fold: the tensors themselves changed
        p0 = items[0][2]
        # ops.mutation_epoch: bumped by everything that writes parameters / BN buffers through raw pointers (b200seg.Adam,
        # the training forward and its CUDA-graph replays) -- those writes do not touch tensor._version
        return (mode, self.dense_impl, v, ops.mutation_epoch(), p0.device, p0.data_ptr(), id(items))

    def _eval_plan(self, mode: str, dense_impl: str):
        """Persistent eval operand buffers + the device table of the one-launch fold/pack kernel
        (b200seg_fold_pack_eval_multi).  Rebuilt only when the parameter tensors themselves are replaced."""
        from ._cabi import lib
        convs = [s for s in self.steps if s.conv is not None]
        ident = tuple(t.data_ptr() for s in convs for m in (s.conv, s.bn) if m is not None
                      for t in list(m.parameters()) + [b for b in m.buffers() if b.is_floating_point()])
        key = (mode, dense_impl, ident)
        plan = getattr(self, "_eval_plan_cache", None)
        if plan is not None and plan["key"] == key:
            return plan
        dev = convs[0].conv.weight.device
        chunk = int(lib.b200seg_fold_chunk())
        tc = dense_impl == "tc"
        packed: Dict[str, dict] = {}
        rows, ct, ci = [], [], []
        mirror_src, mirror_dst, mirrors = [], [], {}
        import struct

        def f32ptr(t):
            """fp32 source of a parameter/buffer: the tensor itself, or (model.bfloat16()) a persistent fp32 mirror that
            is refreshed with one multi-tensor copy before every repack."""
            if t is None:
                return 0
            if t.dtype == torch.float32 and t.is_contiguous():
                return t.data_ptr()
            if id(t) not in mirrors:
                mirrors[id(t)] = torch.empty(t.shape, device=dev, dtype=torch.float32)
                mirror_src.append(t); mirror_dst.append(mirrors[id(t)])
            return mirrors[id(t)].data_ptr()

        def add_row(s, out_w, out_b, kind, ldw):
            w, bn = s.conv.weight, s.bn
            cout, cin, kk = w.shape[0], w.shape[1], w.shape[2] * w.shape[3]
            eps = struct.unpack("<I", struct.pack("<f", float(bn.eps) if bn is not None else 0.0))[0]
            ti = len(rows) // 12
            rows.extend([f32ptr(w), f32ptr(s.conv.bias), f32ptr(bn.weight) if bn is not None else 0,
                         f32ptr(bn.bias) if bn is not None else 0, f32ptr(bn.running_mean) if bn is not None else 0,
                         f32ptr(bn.running_var) if bn is not None else 0,
                         out_w.data_ptr(), 0 if out_b is None else out_b.data_ptr(),
                         (cin << 32) | cout, (ldw << 32) | kk, (eps << 32) | kind, 0])
            n = cout * cin * kk + (cout if out_b is not None else 0)
            for c in range((n + chunk - 1) // chunk):
                ct.append(ti); ci.append(c)

        for s in convs:
            w = s.conv.weight
            cout, cin, kk = w.shape[0], w.shape[1], w.shape[2] * w.shape[3]
            bfull = torch.zeros((cout + 63) // 64 * 64, device=dev, dtype=torch.float32)
            if s.op == "stem":
                ow = torch.zeros(w.shape[2], w.shape[3], cin, cout, device=dev, dtype=torch.float32)
                add_row(s, ow, bfull, 2, 0)
                packed[s.name] = dict(w=ow, b=bfull[:cout])
            elif s.op == "dw":
                ow = torch.zeros(kk, cout, device=dev, dtype=torch.float32)
                add_row(s, ow, bfull, 3, cout)
                packed[s.name] = dict(w=ow, b=bfull[:cout], b64=bfull)
                cep = bfull.numel()
                if mode == "bf16":
                    wdiag = torch.zeros(cout, kk, 64, device=dev, dtype=torch.bfloat16)
                    add_row(s, wdiag, None, 4, 0)
                    packed[s.name]["wdiag"] = wdiag
                    wb = torch.zeros(kk, cout, device=dev, dtype=torch.bfloat16)      # bf16 taps (mixed-precision FMA kernels)
                    add_row(s, wb, None, 5, cout)
                    packed[s.name]["wb"] = wb
                    w64 = wb                                                          # ... zero padded to 64-channel chunks
                    if cep != cout:
                        w64 = torch.zeros(kk, cep, device=dev, dtype=torch.bfloat16)
                        add_row(s, w64, None, 5, cep)
                    packed[s.name]["w64"] = w64
            else:
                cp = max(cout, s.pad_cout) if s.pad_cout else cout
                ow = torch.zeros(cp, kk * cin, device=dev, dtype=torch.bfloat16 if tc else torch.float32)
                add_row(s, ow, bfull, 0 if tc else 1, 0)
                packed[s.name] = dict(w=ow, b=bfull[:cp], b64=bfull)
        if mode == "bf16" and tc:
            # operands of the fused inverted-residual kernel: views of the three layers' packs (parameter vectors are
            # zero padded to the 64-channel chunks the kernel processes)
            for e, d, pj in self._mb_triples():
                cop = (pj.conv.weight.shape[0] + 15) // 16 * 16
                packed[pj.name + "#mb"] = dict(
                    w_exp=packed[e.name]["w"], b_exp=packed[e.name]["b64"], w_dw=packed[d.name]["w64"],
                    b_dw=packed[d.name]["b64"], w_proj=packed[pj.name]["w"], b_proj=packed[pj.name]["b64"][:cop])
        plan = dict(key=key, packed=packed, n=len(ct), mirror_src=mirror_src, mirror_dst=mirror_dst,
                    table=torch.tensor(rows, dtype=torch.int64, device=dev),
                    ct=torch.tensor(ct, dtype=torch.int32, device=dev), ci=torch.tensor(ci, dtype=torch.int32, device=dev))
        self._eval_plan_cache = plan
        self._packed_key = None
        return plan

    def _pack_eval(self, mode: str):
        """Folded + packed eval weights for the current parameter values: ONE kernel launch when anything changed."""
        from ._cabi import check, lib, ptr
        dense_impl = self.dense_impl or ("tc" if mode == "bf16" else "simt")
        key = self._version_key(mode)
        if key == self._packed_key:           # nothing written since the last fold (the steady-state inference call): ~0.1 ms of
            return self._packed               # host time instead of ~1.5 ms for re-deriving the operand plan's identity
        plan = self._eval_plan(mode, dense_impl)
        if key != self._packed_key:
            if plan["mirror_src"]:
                with torch.no_grad():
                    torch._foreach_copy_(plan["mirror_dst"], plan["mirror_src"])
            check(lib.b200seg_fold_pack_eval_multi(ptr(plan["table"]), ptr(plan["ct"]), ptr(plan["ci"]), plan["n"],
                                                   torch.cuda.current_stream().cuda_stream), "fold_pack_eval_multi")
            self._packed, self._packed_key = plan["packed"], key
        return self._packed

    # ------------------------------------------------------------------ fused inverted-residual blocks
    def _mb_triples(self):
        """(expand 1x1, depthwise 3x3, project 1x1) step triples of the encoder's expand-ratio-6 blocks."""
        out = []
        st = self.steps
        for i in range(len(st) - 2):
            e, d, pj = st[i], st[i + 1], st[i + 2]
            if (e.op == "dense" and e.taps == 1 and e.act == ACT_RELU6 and e.res is None and d.op == "dw"
                    and d.src == e.dst and pj.op == "dense" and pj.taps == 1 and pj.src == d.dst
                    and pj.act == ACT_NONE and not pj.pad_cout and (pj.res is None or pj.res == e.src)):
                out.append((e, d, pj))
        return out

    def _schedule(self, mode: str, dense_impl: str, H: int, W: int, in_dtype=torch.float32) -> List[Step]:
        """Eval schedule for an input of H x W: self.steps with the inverted-residual triples replaced by one
        fused step (measured faster for every block, tools/kbench_mb.py), and the output tail by its fused kernel."""
        from ._cabi import lib
        impl = self.mbconv_impl or "auto"
        if mode != "bf16" or dense_impl != "tc":
            return self.steps
        key = (impl, self.tail_impl, self.head_impl, H, W, in_dtype)
        if key not in self._eval_sched:
            first = {id(e): (e, d, pj) for e, d, pj in self._mb_triples()}
            out, skip = [], set()
            scale = {}                       # schedule name -> downscale factor of its tensor w.r.t. the input
            for st in self.steps:
                scale[st.dst] = scale.get(st.src, 1) * (st.stride if st.op in ("stem", "dw") else 1)
                if st.op == "upcat":
                    scale[st.dst] = scale[st.src] // 2
            for st in self.steps:
                if id(st) in skip:
                    continue
                if id(st) in first and impl != "unfused":
                    e, d, pj = first[id(st)]
                    in_w = W // max(scale.get(e.src, 1), 1)
                    # every expand-ratio-6 block is faster fused since the depthwise stencil runs on the mixed-precision FMA
                    # (tools/kbench_mb.py; before, the stride-2 block at half resolution was 5 % slower fused)
                    if impl in ("fused", "auto") or in_w < 0:
                        out.append(Step("mbconv", pj.name.rsplit(".conv.", 1)[0], e.src, pj.dst, stride=d.stride,
                                        res=pj.res, parts=(e, d, pj)))
                        skip.update((id(d), id(pj)))
                        continue
                out.append(st)
            # head of MobileNetV2UNet: features.0 (stem) -> features.1 (depthwise + linear 1x1) as one kernel
            if (self.head_impl != "unfused" and len(out) >= 3 and out[0].op == "stem" and out[1].op == "dw"
                    and out[2].op == "dense" and out[1].src == out[0].dst and out[2].src == out[1].dst
                    and out[0].stride == 2 and out[1].stride == 1 and out[2].taps == 1 and out[2].res is None
                    and out[0].act == ACT_RELU6 and out[1].act == ACT_RELU6 and out[2].act == ACT_NONE and not out[2].pad_cout
                    and in_dtype in (torch.float32, torch.bfloat16)
                    and not any(t.src in (out[0].dst, out[1].dst) or t.res in (out[0].dst, out[1].dst) for t in out[3:])
                    and lib.b200seg_stem_mb1_supported(ops.F32 if in_dtype == torch.float32 else ops.BF16, H, W, out[0].conv.weight.shape[0], out[2].conv.weight.shape[0])):
                st0, dw1, pw1 = out[0], out[1], out[2]
                out = [Step("stem_mb1", "backbone.features.0+1", st0.src, pw1.dst, parts=(st0, dw1, pw1))] + out[3:]
            # output tail of MobileNetV2UNet: outc.conv.0 -> outc.conv.3 -> final_upsample (+ argmax) as one kernel
            if (self.tail_impl != "unfused" and len(out) >= 3 and out[-1].op == "final" and self.out_ch <= 16
                    and out[-2].op == "dense" and out[-3].op == "dense" and out[-2].taps == 1 and out[-3].taps == 1
                    and tuple(out[-3].conv.weight.shape[:2]) == (16, 32) and out[-2].conv.weight.shape[1] == 16):
                c0, c3, fin = out[-3], out[-2], out[-1]
                out = out[:-3] + [Step("tail", "outc+final_upsample", c0.src, fin.dst, parts=(c0, c3, fin))]
            self._eval_sched[key] = out
        return self._eval_sched[key]

    # ------------------------------------------------------------------ helpers
    def _mode(self, x: torch.Tensor) -> str:
        if self.precision is not None:
            return self.precision
        p0 = next(self.model.parameters())
        if p0.dtype == torch.bfloat16:
            return "bf16"
        if torch.is_autocast_enabled() and torch.get_autocast_dtype("cuda") == torch.bfloat16:
            return "bf16"
        if p0.dtype != torch.float32:
            raise TypeError(f"b200seg supports float32 and bfloat16 modules, got {p0.dtype}")
        return "fp32"

    def _check_input(self, x):
        if x.dim() != 4 or x.shape[1] != 3:
            raise ValueError(f"expected input [B,3,H,W], got {tuple(x.shape)}")
        B, _, H, W = x.shape
        if B == 0:
            raise ValueError("empty batch")
        d = self.divisor
        if H % d or W % d:
            # the reference itself fails at torch.cat for such sizes (unet.py:103; SURVEY finding 8)
            raise ValueError(f"H and W must be multiples of {d} (got {H}x{W}); pad the frame first")
        p0 = next(self.model.parameters())
        if p0.device != x.device:
            raise RuntimeError(f"input on {x.device} but model on {p0.device}")

    # ------------------------------------------------------------------ forward (eval)
    def _run_step(self, s: Step, env, pk, mode: str, sdt, dense_impl: str, out_dtype, want_mask: bool, metrics=None, out=None):
        """Launch the kernel of one fused step; inputs/outputs live in ``env`` by schedule name.  ``out``: existing output
        buffer (only for the head step, which is launched outside the captured graph into a static buffer).  ``metrics``:
        (SegmentationMetrics, target): the last step accumulates validation metrics instead of writing an output."""
        if s.op == "stem":
            p = pk[s.name]
            env[s.dst] = ops.conv3x3_smallcin(env[s.src], p["w"], p["b"], s.stride, s.act, sdt, out=out)
        elif s.op == "dw":
            p = pk[s.name]
            if mode == "bf16" and self.dw_impl == "tc":
                env[s.dst] = ops.dwconv3x3_tc(env[s.src], p["wdiag"], p["b"], s.stride, s.act, flags=self.tc_flags)
            elif mode == "bf16" and self.dw_impl != "simt":
                # bf16 taps + mixed-precision FMA (FHFMA.BF16): 15-25 % faster than the f32-tap kernel on stride 1 and faster
                # than the block-diagonal tensor-core variant on every layer of this net (tools/kbench_dw.py)
                env[s.dst] = ops.dwconv3x3_bf16w(env[s.src], p["wb"], p["b"], s.stride, s.act)
            else:
                env[s.dst] = ops.dwconv3x3(env[s.src], p["w"], p["b"], s.stride, s.act)
        elif s.op == "dense":
            p = pk[s.name]
            res = env[s.res] if s.res else None
            if dense_impl == "tc":
                env[s.dst] = ops.conv_tc(env[s.src], p["w"], p["b"], s.taps, s.act, res, flags=self.tc_flags)
            else:
                env[s.dst] = ops.conv_simt(env[s.src], p["w"], p["b"], s.taps, s.act, res)
        elif s.op == "stem_mb1":
            p0, p1, p2 = (pk[q.name] for q in s.parts)
            env[s.dst] = ops.stem_mb1(env[s.src], p0["w"], p0["b"], p1["wb"], p1["b"], p2["w"], p2["b"], out=out)
        elif s.op == "mbconv":
            p = pk[s.parts[2].name + "#mb"]
            env[s.dst] = ops.mbconv(env[s.src], p["w_exp"], p["b_exp"], p["w_dw"], p["b_dw"], p["w_proj"], p["b_proj"],
                                    s.stride, s.res is not None, flags=self.mbconv_flags)
        elif s.op == "tail" and metrics is not None:
            p0, p3 = pk[s.parts[0].name], pk[s.parts[1].name]
            sm, tgt = metrics
            ops.tail_fused_metrics(env[s.src], p0["w"], p0["b64"], p3["w"], p3["b64"], self.out_ch, tgt, sm.ignore_index,
                                   sm.confusion, sm.counts, sm.loss_sum)
            env[s.dst] = None
        elif s.op == "tail":
            p0, p3 = pk[s.parts[0].name], pk[s.parts[1].name]
            env[s.dst] = ops.tail_fused(env[s.src], p0["w"], p0["b64"], p3["w"], p3["b64"], self.out_ch, out_dtype, want_mask, out=out)
        elif s.op == "upcat":
            env[s.dst] = ops.upsample2x_concat(env[s.res], env[s.src])
        elif s.op == "pool":
            env[s.dst] = ops.maxpool2x2(env[s.src])
        elif s.op in ("final", "to_nchw") and metrics is not None:
            sm, tgt = metrics
            if s.op == "final":      # f32 NCHW logits: the values the argmax of predict_mask compares
                ops.seg_metrics(ops.upsample2x_ac_nchw(env[s.src], self.out_ch, torch.float32), tgt, self.out_ch,
                                sm.ignore_index, sm.confusion, sm.counts, sm.loss_sum)
            else:                    # UNet: straight from the NHWC logits buffer, no layout pass
                ops.seg_metrics(env[s.src], tgt, self.out_ch, sm.ignore_index, sm.confusion, sm.counts, sm.loss_sum, nhwc=True)
            env[s.dst] = None
        elif s.op == "final":
            if want_mask:
                env[s.dst] = ops.upsample2x_ac_argmax(env[s.src], self.out_ch, out=out)
            else:
                env[s.dst] = ops.upsample2x_ac_nchw(env[s.src], self.out_ch, out_dtype, out=out)
        elif s.op == "to_nchw":
            if want_mask:
                env[s.dst] = ops.nhwc_argmax(env[s.src], self.out_ch, out=out)
            else:
                env[s.dst] = ops.nhwc_to_nchw(env[s.src], self.out_ch, out_dtype, out=out)
        else:  # pragma: no cover
            raise AssertionError(s.op)

    @torch.no_grad()
    def forward_eval(self, x: torch.Tensor, want_mask: bool = False, keep: Optional[dict] = None,
                     profile: Optional[list] = None, out=None, metrics=None):
        """Eval-mode forward.  ``keep`` (dict) receives every intermediate NHWC tensor by schedule name;
        ``profile`` (list) receives (step, start_event, end_event, bytes, flops) per launched kernel.
        ``metrics`` = (SegmentationMetrics, target): the last step accumulates the validation metrics and returns None.

        Steady state (same shape seen ``graph_after`` times, weights unchanged): the first kernel (reads the
        caller's NCHW tensor) and the last one (writes a fresh NCHW result) are launched directly, every
        kernel in between is replayed from ONE captured CUDA graph over static activation buffers, so a
        forward costs three launches of host time instead of ~70."""
        self._check_input(x)
        mode = self._mode(x)
        sdt = torch.bfloat16 if mode == "bf16" else torch.float32
        dense_impl = self.dense_impl or ("tc" if mode == "bf16" else "simt")
        if dense_impl == "tc" and mode != "bf16":
            raise RuntimeError("tensor-core convs need bf16 storage")
        pk = self._pack_eval(mode)
        if x.dtype not in (torch.float32, torch.bfloat16):
            raise TypeError(f"input dtype {x.dtype} not supported")
        x = x.contiguous()
        out_dtype = x.dtype
        args = (pk, mode, sdt, dense_impl, out_dtype, want_mask, metrics)
        steps = self._schedule(mode, dense_impl, x.shape[2], x.shape[3], x.dtype)

        if keep is None and profile is None and self.use_graphs and not torch.cuda.is_current_stream_capturing():
            key = (tuple(x.shape), x.dtype, mode, dense_impl, self.dw_impl, self.mbconv_impl, self.tail_impl, self.head_impl, self.tc_flags,
                   self.mbconv_flags, self._packed_key, x.device)
            ent = self._graphs.get(key)
            if ent is None:
                if len(self._graphs) >= 3:
                    self._graphs.clear()            # weights or shapes keep changing: do not hoard pools
                ent = self._graphs[key] = {"seen": 0, "graph": None}
            ent["seen"] += 1
            if ent["graph"] is None and ent["seen"] > self.graph_after:
                self._capture(ent, x, args, steps)
            if ent["graph"] is not None:
                env = {"x": x}
                self._run_step(ent["head"], env, *args, out=ent["head_out"])
                ent["graph"].replay()
                env[ent["tail"].src] = ent["body_out"]
                self._run_step(ent["tail"], env, *args, out=out)
                return env["out"]

        env: Dict[str, Optional[torch.Tensor]] = {"x": x}
        for s in steps:
            if profile is not None:
                ev0 = torch.cuda.Event(enable_timing=True); ev0.record()
            self._run_step(s, env, *args, out=out if s is steps[-1] else None)
            if profile is not None:
                ev1 = torch.cuda.Event(enable_timing=True); ev1.record()
                nbytes, flops = self.step_cost(s, env, pk)
                profile.append((s, ev0, ev1, nbytes, flops))
        if keep is not None:
            keep.update(env)
        return env["out"]

    def _capture(self, ent, x, args, steps):
        """Capture steps[1:-1] into a CUDA graph.  Buffers allocated inside the capture come from the
        graph's private pool and stay valid for every replay."""
        pk, mode, sdt, dense_impl, out_dtype, want_mask, metrics = args
        head, body, tail = steps[0], steps[1:-1], steps[-1]
        assert head.op in ("stem", "stem_mb1") and tail.op in ("final", "to_nchw", "tail")
        ent["head"] = head
        env = {"x": x}
        self._run_step(head, env, *args)
        ent["head_out"] = env[head.dst]
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for s in body:
                self._run_step(s, env, *args)
        ent["graph"], ent["body_out"], ent["tail"] = g, env[tail.src], tail
        ent["env"] = env          # keeps the captured buffers referenced

    # ------------------------------------------------------------------ cost model
    @staticmethod
    def layer_model_bytes(s: Step, env, pk) -> int:
        """Bytes of the step under SURVEY 8(d)'s per-LAYER traffic model ("each conv(+BN+act[+res]) reads its input once and
        writes its output once in the storage dtype", i.e. the figure behind its 115.7 MB/img): for a kernel that fuses
        several layers this is the SUM over the layers it replaces -- the intermediates it keeps on chip are counted, which
        is why a fused kernel may exceed 1.0 of the HBM roofline on this scale.  Equal to step_cost()[0] for unfused steps."""
        fused_io, _ = Engine.step_cost(s, env, pk)
        out = env[s.dst]
        esz = 2                                            # bf16 storage of every intermediate (fused steps are bf16-only)
        if s.op == "mbconv":
            e, d, pj = s.parts
            ce = e.conv.weight.shape[0]
            npix_in = env[s.src].numel() // env[s.src].shape[-1]
            npix_out = out.numel() // out.shape[-1]
            return fused_io + esz * ce * (2 * npix_in + 2 * npix_out)      # expand out + dw in, dw out + project in
        if s.op == "stem_mb1":
            cs = s.parts[0].conv.weight.shape[0]
            npix = out.numel() // out.shape[-1]
            return fused_io + esz * cs * 4 * npix                          # stem out + dw in, dw out + 1x1 in
        if s.op == "tail":
            c0, c3, _ = s.parts
            npix = env[s.src].numel() // env[s.src].shape[-1]
            mid, cls = c0.conv.weight.shape[0], c3.conv.weight.shape[0]
            return fused_io + esz * npix * (2 * mid + 2 * cls)             # outc.0 out + outc.3 in, logits out + upsample in
        return fused_io

    @staticmethod
    def step_cost(s: Step, env, pk):
        """Algorithmic HBM bytes and FLOPs of one fused step (SURVEY 8d traffic model): read every
        input once, write the output once, weights once; FLOPs = 2*MAC."""
        out = env[s.dst]
        nbytes = out.numel() * out.element_size() + env[s.src].numel() * env[s.src].element_size()
        flops = 0
        if s.op == "tail":
            c0, c3, _ = s.parts
            npix = env[s.src].numel() // env[s.src].shape[-1]
            nbytes += (c0.conv.weight.numel() + c3.conv.weight.numel()) * 2 + 2 * 16 * 4
            return nbytes, 2 * npix * (c0.conv.weight.numel() + c3.conv.weight.numel())
        if s.op == "stem_mb1":
            st0, dw1, pw1 = s.parts
            cs, co = st0.conv.weight.shape[0], pw1.conv.weight.shape[0]
            npix = out.numel() // out.shape[-1]
            nbytes += 27 * cs * 4 + 9 * cs * 2 + co * cs * 2 + (2 * cs + co) * 4
            return nbytes, 2 * npix * (27 * cs + 9 * cs + cs * co)
        if s.op == "mbconv":
            # algorithmic bytes of the FUSED block: input, output, residual and the three weight sets once
            e, d, pj = s.parts
            p = pk[pj.name + "#mb"]
            ce = e.conv.weight.shape[0]
            npix_in = env[s.src].numel() // env[s.src].shape[-1]
            npix_out = out.numel() // out.shape[-1]
            if s.res:
                nbytes += env[s.res].numel() * env[s.res].element_size()
            nbytes += (p["w_exp"].numel() + p["w_proj"].numel() + 9 * ce) * 2 + (2 * ce + out.shape[-1]) * 4
            flops = 2 * (npix_in * ce * env[s.src].shape[-1] + npix_out * ce * 9 + npix_out * ce * out.shape[-1])
            return nbytes, flops
        if s.res:
            nbytes += env[s.res].numel() * env[s.res].element_size()
        if s.conv is not None:
            p = pk[s.name]
            nbytes += p["w"].numel() * p["w"].element_size() + p["b"].numel() * 4
            if s.op == "dw":
                nbytes -= p["w"].numel() * p["w"].element_size() - 9 * out.shape[-1] * 2   # 9 taps/channel are the algorithmic weights
                flops = 2 * 9 * out.numel()
            elif s.op == "stem":
                flops = 2 * out.numel() * 27
            else:
                cout = s.conv.weight.shape[0]                      # real (unpadded) output channels
                flops = 2 * (out.numel() // out.shape[-1]) * cout * s.taps * env[s.src].shape[-1]
        return nbytes, flops

    # ------------------------------------------------------------------ dispatch
    def forward(self, x: torch.Tensor, want_mask: bool = False, out=None, metrics=None):
        # every kernel is launched on the current stream of the CURRENT device: make the input's device current for the
        # whole call (model.to("cuda:1") while cuda:0 is current must work like any nn.Module)
        with torch.cuda.device(x.device):
            if self.model.training:
                if want_mask:
                    raise RuntimeError("predict_mask needs model.eval()")
                if metrics is not None:
                    raise RuntimeError("evaluate needs model.eval()")
                from . import train_path
                return train_path.forward_train(self, x)
            return self.forward_eval(x, want_mask, out=out, metrics=metrics)
