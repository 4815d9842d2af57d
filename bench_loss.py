"""Cross-entropy benchmark: b200seg.CrossEntropyLoss with torch's options against the default fused loss and against
torch.nn.functional.cross_entropy, at the training step's shape: B = 32, C = 10, 256x512 f32 logits (168 MB, larger than
the 126 MB L2), seeded logits and labels (5 % ignored).

Legs (forward + backward to d(logits), CUDA events over --steps calls after --warmup untimed ones, rounds alternate legs):
  1 default            CrossEntropyLoss()(z, t_int64).backward()
  2 weight_ls          weight + label_smoothing=0.1, int64 targets ('mean': weighted count + one fused pass)
  3 weight_ls_u8       (2) with uint8 targets and ignore_index=255
  4 none               reduction='none', weight + label_smoothing=0.1: loss map, then backward with a per-pixel gout
  5 torch_weight_ls    F.cross_entropy with the arguments of (2)
  5 torch_none         F.cross_entropy with the arguments of (4)
  6 train_default      one MobileNetV2UNet(10) training step, bf16 activations, b200seg.Adam, default loss
  6 train_options      the same step with the loss of (3)

The kernel section times the tensor-level wrappers without autograd, replayed from a CUDA graph (device time only).
Bytes are taken from shapes: logits read and d(logits) written (4 B each per element), targets (8 or 1 B per pixel), and
for (4) the loss map and gout (4 B per pixel each).  They are set against 7.7 TB/s, the data-sheet HBM3e bandwidth of one
B200.  The device name and its enforced power limit are read in the same run.

    python bench_loss.py [--steps 50] [--warmup 5] [--rounds 5] [--train-steps 10] [--out result.json]
"""
import argparse
import json
import os
import statistics
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [ROOT, os.path.join(ROOT, "team02-objectdetection_b200")]

from bench_eval import _device_info  # noqa: E402

B, NCLS, H, W = 32, 10, 256, 512
HBM_BW = 7.7e12          # B/s, NVIDIA HGX B200 data sheet, one GPU


def _time(fn, n):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n        # ms per call


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--train-steps", type=int, default=10)
    ap.add_argument("--no-train", action="store_true", help="skip the training-step legs")
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_loss.py needs a CUDA device")
    import b200seg

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    g = torch.Generator(device="cpu").manual_seed(0)
    z = (torch.randn(B, NCLS, H, W, generator=g) * 3).to(dev).requires_grad_()
    t = torch.randint(0, NCLS, (B, H, W), generator=g)
    ign = torch.rand(B, H, W, generator=g) < 0.05
    t64 = torch.where(ign, torch.full_like(t, -100), t).to(dev)
    t8 = torch.where(ign, torch.full_like(t, 255), t).to(torch.uint8).to(dev)
    w = (torch.rand(NCLS, generator=g) + 0.5).to(dev)
    gout = torch.randn(B, H, W, generator=g).to(dev)

    crit = {
        "1_default": b200seg.CrossEntropyLoss(),
        "2_weight_ls": b200seg.CrossEntropyLoss(weight=w, label_smoothing=0.1),
        "3_weight_ls_u8": b200seg.CrossEntropyLoss(weight=w, ignore_index=255, label_smoothing=0.1),
        "4_none": b200seg.CrossEntropyLoss(weight=w, label_smoothing=0.1, reduction="none"),
    }

    def mean_leg(c, tg):
        def f():
            z.grad = None
            c(z, tg).backward()
        return f

    def none_leg(lossfn, tg):
        def f():
            z.grad = None
            lossfn(z, tg).backward(gout)
        return f

    def torch_mean(zz, tg):
        return F.cross_entropy(zz, tg, weight=w, label_smoothing=0.1)

    def torch_none(zz, tg):
        return F.cross_entropy(zz, tg, weight=w, label_smoothing=0.1, reduction="none")

    n_el, n_px = B * NCLS * H * W, B * H * W
    legs = {
        "1_default": (mean_leg(crit["1_default"], t64), 8 * n_el + 8 * n_px),
        "2_weight_ls": (mean_leg(crit["2_weight_ls"], t64), 8 * n_el + 8 * n_px),
        "3_weight_ls_u8": (mean_leg(crit["3_weight_ls_u8"], t8), 8 * n_el + n_px),
        "4_none": (none_leg(crit["4_none"], t64), 8 * n_el + 8 * n_px + 8 * n_px),
        "5_torch_weight_ls": (mean_leg(torch_mean, t64), 8 * n_el + 8 * n_px),
        "5_torch_none": (none_leg(torch_none, t64), 8 * n_el + 8 * n_px + 8 * n_px),
    }
    res = {"device": _device_info(dev), "shape": [B, NCLS, H, W], "logits_MB": round(4 * n_el / 1e6, 1),
           "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds, "legs": {}}

    # the option paths compute what torch computes (one batch, before timing)
    z64 = z.detach().double().requires_grad_()
    ref = F.cross_entropy(z64, t64, weight=w.double(), label_smoothing=0.1)
    ref.backward()
    got = {}
    for name in ("2_weight_ls", "3_weight_ls_u8"):
        z.grad = None
        loss = crit[name](z, t64 if name == "2_weight_ls" else t8)
        loss.backward()
        got[name] = {"loss_rel_err": abs(float(loss) - float(ref)) / abs(float(ref)),
                     "grad_err_over_max": float((z.grad.double() - z64.grad).abs().max() / z64.grad.abs().max())}
    res["check_vs_torch_f64"] = got

    for name, (fn, _) in legs.items():
        for _ in range(args.warmup):
            fn()
    times = {name: [] for name in legs}
    for _ in range(args.rounds):
        for name, (fn, _) in legs.items():
            times[name].append(_time(fn, args.steps))
    for name, (_, nbytes) in legs.items():
        ms = statistics.median(times[name])
        res["legs"][name] = {"ms": round(ms, 4), "ms_all_rounds": [round(v, 4) for v in times[name]], "bytes": int(nbytes),
                             "TB_per_s": round(nbytes / (ms * 1e-3) / 1e12, 2),
                             "hbm_fraction": round(nbytes / (ms * 1e-3) / HBM_BW, 3)}
    L = res["legs"]
    one_pass_ms = 4 * n_el / HBM_BW * 1e3
    res["ratios"] = {
        "2_over_1": round(L["2_weight_ls"]["ms"] / L["1_default"]["ms"], 3),
        "3_over_1": round(L["3_weight_ls_u8"]["ms"] / L["1_default"]["ms"], 3),
        "4_minus_1_ms": round(L["4_none"]["ms"] - L["1_default"]["ms"], 4),
        "one_logits_pass_at_datasheet_ms": round(one_pass_ms, 4),
        "torch_weight_ls_over_2": round(L["5_torch_weight_ls"]["ms"] / L["2_weight_ls"]["ms"], 2),
        "torch_none_over_4": round(L["5_torch_none"]["ms"] / L["4_none"]["ms"], 2),
    }
    del z64, ref

    # kernel section: the C-ABI wrappers alone (no autograd; a memset, the count kernel when 'mean', the loss kernel, a few
    # scalar ops), --steps calls captured in one CUDA graph and replayed, so the time is the device's, not the host's
    from b200seg import ops
    zk = z.detach()
    kern = {
        "default_count_fwd_grad": (lambda: ops.softmax_ce(zk, t64), 8 * n_el + 16 * n_px),
        "options_count_fwd_grad": (lambda: ops.softmax_ce_ex(zk, t64, w, -100, 0.1, "mean"), 8 * n_el + 16 * n_px),
        "options_u8_count_fwd_grad": (lambda: ops.softmax_ce_ex(zk, t8, w, 255, 0.1, "mean"), 8 * n_el + 2 * n_px),
        "none_fwd_map": (lambda: ops.softmax_ce_ex(zk, t64, w, -100, 0.1, "none"), 4 * n_el + 12 * n_px),
        "none_bwd": (lambda: ops.softmax_ce_ex_backward(zk, t64, gout, w, -100, 0.1), 8 * n_el + 12 * n_px),
    }
    res["kernels"] = {}
    for name, (fn, nbytes) in kern.items():
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(args.warmup):
                fn()
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for _ in range(args.steps):
                fn()
        graph.replay()
        ms = statistics.median(_time(graph.replay, 1) for _ in range(args.rounds)) / args.steps
        del graph
        res["kernels"][name] = {"us": round(ms * 1e3, 1), "bytes": int(nbytes), "TB_per_s": round(nbytes / (ms * 1e-3) / 1e12, 2),
                                "hbm_fraction": round(nbytes / (ms * 1e-3) / HBM_BW, 3)}

    if not args.no_train:
        model = b200seg.MobileNetV2UNet(output_channels=NCLS).to(dev)
        eng = model._get_engine()
        eng.precision = "bf16"
        opt = b200seg.Adam(model.parameters(), lr=1.5e-4)
        model.train()
        x = torch.randn(B, 3, H, W, generator=g).to(dev)
        z.grad = None

        def train_leg(c, tg):
            def f():
                opt.zero_grad()
                c(model(x), tg).backward()
                opt.step()
            return f

        tlegs = {"6_train_default": train_leg(crit["1_default"], t64), "6_train_options": train_leg(crit["3_weight_ls_u8"], t8)}
        for fn in tlegs.values():
            for _ in range(max(args.warmup, eng.graph_after + 2)):
                fn()
        tt = {name: [] for name in tlegs}
        for _ in range(args.rounds):
            for name, fn in tlegs.items():
                tt[name].append(_time(fn, args.train_steps))
        for name in tlegs:
            res["legs"][name] = {"ms": round(statistics.median(tt[name]), 3), "ms_all_rounds": [round(v, 3) for v in tt[name]],
                                 "img_per_s": round(B / (statistics.median(tt[name]) * 1e-3), 1)}
        res["ratios"]["6_options_over_default"] = round(L["6_train_options"]["ms"] / L["6_train_default"]["ms"], 4)
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
