"""Validation benchmark: MobileNetV2UNet(10) in bf16, eval mode, batch 64 at 3x256x512, seeded weights, inputs and labels.

Legs (img/s from CUDA events over --steps calls after --warmup untimed ones, 4 rotating batches resident in HBM):
  a  model.evaluate(x, t_int64, metrics)   loss + argmax + confusion in the output-tail kernel; no logits tensor
  b  model.evaluate(x, t_uint8, metrics)   the same with 8.4 MB of uint8 labels instead of 67 MB of int64
  c  model(x) + metrics.update(logits, t)  f32 NCHW logits written, then the standalone metrics kernel
  d  model(x) + the plain torch loop       F.cross_entropy(sum) + argmax + bincount over a boolean mask (host syncs)
  e  model.predict_mask(x)                 the floor: the same network with the argmax-only tail

Inputs are f32 NCHW (the model's public input; the bf16 engine runs on them), so the logits of legs c / d are the f32 values
the fused tail compares and all four metric legs must give the same confusion matrix -- asserted on one batch.  The kernel
section times the output-tail kernel alone in its three epilogues on one decoder output, and the standalone metrics kernel,
each over 50 back-to-back launches; HBM bytes are computed from shapes (decoder output, targets, logits / mask written)
and set against 7.7 TB/s, the data-sheet HBM3e bandwidth of one B200.  The working set of each kernel (>= 142 MB) is
larger than the 126 MB L2.  The device name and its enforced power limit are read through NVML in the same run.

    python bench_eval.py [--steps 20] [--warmup 5] [--batch 64] [--out result.json]
"""
import argparse
import json
import os
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [ROOT, os.path.join(ROOT, "team02-objectdetection_b200")]

NCLS, H, W = 10, 256, 512
HBM_BW = 7.7e12          # B/s, NVIDIA HGX B200 data sheet, one GPU


def _device_info(dev):
    info = {"name": torch.cuda.get_device_name(dev), "power_limit_w": None}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(dev.index or 0)
        info["power_limit_w"] = pynvml.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0
        info["nvml_name"] = pynvml.nvmlDeviceGetName(h)
        if isinstance(info["nvml_name"], bytes):
            info["nvml_name"] = info["nvml_name"].decode()
        pynvml.nvmlShutdown()
    except Exception as e:  # noqa: BLE001 -- reported, not hidden
        info["nvml_error"] = repr(e)
    return info


def _time(fn, n, warmup):
    for i in range(warmup):
        fn(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3          # seconds


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_eval.py needs a CUDA device")
    import b200seg
    from b200seg import ops

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B = args.batch
    torch.manual_seed(0)
    model = b200seg.MobileNetV2UNet(output_channels=NCLS).to(dev).bfloat16().eval()
    eng = model._get_engine()
    g = torch.Generator(device="cpu").manual_seed(0)
    nrot = 4
    xs = [torch.randn(B, 3, H, W, generator=g).to(dev) for _ in range(nrot)]
    ts = []
    for _ in range(nrot):
        t = torch.randint(0, NCLS, (B, H, W), generator=g)
        t[torch.rand(B, H, W, generator=g) < 0.05] = -100                   # ignored pixels
        ts.append(t.to(dev))
    t8s = [torch.where(t < 0, torch.full_like(t, 255), t).to(torch.uint8) for t in ts]
    m64 = b200seg.SegmentationMetrics(NCLS, device=dev)
    m8 = b200seg.SegmentationMetrics(NCLS, device=dev, ignore_index=255)
    mc = b200seg.SegmentationMetrics(NCLS, device=dev)
    torch_state = {}

    def torch_loop(logits, t, st):
        v = (t >= 0) & (t < NCLS)
        st["loss"] = st.get("loss", 0.0) + F.cross_entropy(logits, t, reduction="sum")
        pred = logits.argmax(1)
        cm = torch.bincount(t[v] * NCLS + pred[v], minlength=NCLS * NCLS).view(NCLS, NCLS)
        st["cm"] = st.get("cm", 0) + cm

    legs = {
        "a_evaluate_int64": lambda i: model.evaluate(xs[i % nrot], ts[i % nrot], m64),
        "b_evaluate_uint8": lambda i: model.evaluate(xs[i % nrot], t8s[i % nrot], m8),
        "c_forward_update": lambda i: mc.update(model(xs[i % nrot]), ts[i % nrot]),
        "d_forward_torch_loop": lambda i: torch_loop(model(xs[i % nrot]), ts[i % nrot], torch_state),
        "e_predict_mask": lambda i: model.predict_mask(xs[i % nrot]),
    }
    res = {"device": _device_info(dev), "batch": B, "shape": [3, H, W], "classes": NCLS, "input_dtype": "float32",
           "model": "MobileNetV2UNet(10), module .bfloat16(), eval", "steps": args.steps, "warmup": args.warmup, "legs": {}}
    with torch.no_grad():
        for name, fn in legs.items():
            sec = _time(fn, args.steps, args.warmup)
            res["legs"][name] = {"img_per_s": round(B * args.steps / sec, 1), "ms_per_batch": round(sec / args.steps * 1e3, 3)}

        # the four metric legs on one batch: the same confusion matrix
        cms = {}
        state_of = {"a_evaluate_int64": m64, "b_evaluate_uint8": m8, "c_forward_update": mc}
        for name in list(legs)[:4]:
            for m in state_of.values():
                m.reset()
            torch_state.clear()
            legs[name](0)
            cms[name] = state_of[name].confusion.cpu() if name in state_of else torch_state["cm"].cpu()
        ref = cms["a_evaluate_int64"]
        res["confusion_equal_across_legs"] = all(torch.equal(ref, c) for c in cms.values())
        assert res["confusion_equal_across_legs"], {k: (c - ref).abs().sum().item() for k, c in cms.items()}
        res["valid_pixels_one_batch"] = int(ref.sum())

        # kernel section: the output tail in its three epilogues, and the standalone metrics kernel
        env = {}
        eng.forward_eval(xs[0], keep=env)
        tail = [s for s in eng._schedule("bf16", "tc", H, W, torch.float32) if s.op == "tail"][0]
        pk = eng._pack_eval("bf16")
        p0, p3 = pk[tail.parts[0].name], pk[tail.parts[1].name]
        dec = env[tail.src]                                                  # NHWC bf16 [B,128,256,32]
        logits = torch.empty(B, NCLS, H, W, device=dev)
        mask = torch.empty(B, H, W, device=dev, dtype=torch.uint8)
        dec_bytes = dec.numel() * dec.element_size()
        kern = {
            "tail_metrics_int64": (lambda i: ops.tail_fused_metrics(dec, p0["w"], p0["b64"], p3["w"], p3["b64"], NCLS, ts[0], -100,
                                                                    m64.confusion, m64.counts, m64.loss_sum),
                                   dec_bytes + ts[0].numel() * 8),
            "tail_metrics_uint8": (lambda i: ops.tail_fused_metrics(dec, p0["w"], p0["b64"], p3["w"], p3["b64"], NCLS, t8s[0], 255,
                                                                    m8.confusion, m8.counts, m8.loss_sum),
                                   dec_bytes + t8s[0].numel()),
            "tail_mask": (lambda i: ops.tail_fused(dec, p0["w"], p0["b64"], p3["w"], p3["b64"], NCLS, None, True, out=mask),
                          dec_bytes + mask.numel()),
            "tail_logits_f32": (lambda i: ops.tail_fused(dec, p0["w"], p0["b64"], p3["w"], p3["b64"], NCLS, torch.float32, False,
                                                         out=logits), dec_bytes + logits.numel() * 4),
            "seg_metrics_f32_nchw_int64": (lambda i: ops.seg_metrics(logits, ts[0], NCLS, -100, mc.confusion, mc.counts, mc.loss_sum),
                                           logits.numel() * 4 + ts[0].numel() * 8),
        }
        res["kernels"] = {}
        for name, (fn, nbytes) in kern.items():
            sec = _time(fn, 50, 5) / 50
            res["kernels"][name] = {"us": round(sec * 1e6, 1), "bytes": int(nbytes),
                                    "TB_per_s": round(nbytes / sec / 1e12, 2), "hbm_fraction": round(nbytes / sec / HBM_BW, 3)}
    L = res["legs"]
    res["evaluate_int64_vs_predict_mask"] = round(L["a_evaluate_int64"]["img_per_s"] / L["e_predict_mask"]["img_per_s"], 3)
    res["evaluate_int64_vs_torch_loop"] = round(L["a_evaluate_int64"]["img_per_s"] / L["d_forward_torch_loop"]["img_per_s"], 3)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
