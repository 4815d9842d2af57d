"""Object-detection frame loop benchmark: the reference's inference loop (inference.py) with its post-processing on the GPU.

Set-up: MobileNetV2UNet(10) in bf16 with the trained F2 weights (tests/golden/f2_weights.npz), batches of 64 uint8 BGR
frames of 960x540 (the size of the reference's sample video) rendered from oracle.unet_oracle.road_scene_batch, network input
512x256, classes 1..9, close 5, min_area 0.  Two batches rotate, resident in HBM (frames 2 x 99.5 MB, more than the 126 MB L2).

Legs (frames/s and ms per batch from CUDA events over --steps calls after --warmup untimed ones):
  a  preprocess_image + predict_mask                           the floor: frames in, class mask out
  b  a + detect_objects + device-to-host copy of count / stats the boxes on the host (pinned buffer, one copy)
  c  b + overlay(frames, mask, palette, 0.7, 0.3)              plus the blended BGR image
  d  detect_objects alone on the masks of leg a
  e  detect_objects alone on a noise mask (~28 k components per frame)
The cv2 recipe (nearest resize, then per class a 5x5 close and connectedComponentsWithStats) is timed on the host cores for
--cv2-frames frames of the same masks, and its rows are compared with detect_objects' for those frames.  A separate profiler
pass lists the kernel times of detect_objects.  Bytes are computed from the shapes (see _bytes) and set against 7.7 TB/s,
the data-sheet HBM3e bandwidth of one B200.  The device name and enforced power limit are read through NVML in the same run.

    python bench_detect.py [--steps 20] [--warmup 5] [--batch 64] [--out result.json]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.dont_write_bytecode = True            # the tree may be read-only; nothing is cached there
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [ROOT, os.path.join(ROOT, "team02-objectdetection_b200"), os.path.join(ROOT, "tests")]

from bench_eval import HBM_BW, _device_info, _time  # noqa: E402

FW, FH = 960, 540           # frame size (cv2 order: width, height)
NW, NH = 512, 256           # network input
CLASSES = list(range(1, 10))
CLOSE = 5


def _frames(n, seed):
    """uint8 BGR frames [n,540,960,3] rendered from the road-scene generator (the normalised image mapped back to 0..255)."""
    from oracle import unet_oracle as O
    out = np.empty((n, FH, FW, 3), np.uint8)
    mean, std = np.asarray(O.ROAD_MEAN, np.float32), np.asarray(O.ROAD_STD, np.float32)
    for i in range(0, n, 8):
        x, _ = O.road_scene_batch(min(8, n - i), FH, FW, seed=seed * 1000 + i)
        rgb = x.numpy().transpose(0, 2, 3, 1) * std + mean
        out[i:i + 8] = np.clip(np.rint(rgb * 255.0), 0, 255).astype(np.uint8)[..., ::-1]
    return torch.from_numpy(out)


def _bytes(B, Hm, Wm, K, M):
    """HBM bytes detect_objects must move at least, from the shapes: the mask read, the closed bitmask (2 B per pixel) written
    once and read by the four block passes (merge, compress, number, stats), and the rows written.  The union-find parents,
    component ids and statistics scale with the objects, not the frame, and are not counted."""
    px = B * FH * FW
    return B * Hm * Wm + 5 * 2 * px + B * M * 44 + 4 * B


def _cv2_recipe(mask_np, n):
    import cv2
    rows, t0 = [], time.perf_counter()
    for m in mask_np[:n]:
        r = cv2.resize(m, (FW, FH), interpolation=cv2.INTER_NEAREST)
        fr = []
        for c in CLASSES:
            p = cv2.morphologyEx((r == c).astype(np.uint8), cv2.MORPH_CLOSE, np.ones((CLOSE, CLOSE), np.uint8))
            _, _, st, cen = cv2.connectedComponentsWithStats(p, connectivity=8)
            fr += [(c, l) + tuple(int(v) for v in st[l, :5]) + (float(cen[l, 0]), float(cen[l, 1])) for l in range(1, st.shape[0])]
        rows.append(fr)
    sec = time.perf_counter() - t0
    return rows, sec, cv2.getNumThreads()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--cv2-frames", type=int, default=16)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_detect.py needs a CUDA device")
    import b200seg
    from oracle import unet_oracle as O
    from util import expand_aliases, gold

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B = args.batch
    m = b200seg.MobileNetV2UNet(output_channels=10)
    full = dict(m.state_dict())
    full.update(expand_aliases(O.f2_state_dict(gold("f2_weights.npz"))))
    m.load_state_dict(full, strict=True)
    model = m.to(dev).bfloat16().eval()
    nrot = 2
    frames = [_frames(B, seed=s).to(dev) for s in range(nrot)]
    xn = [torch.empty(B, 3, NH, NW, device=dev, dtype=torch.bfloat16) for _ in range(nrot)]
    masks = [torch.empty(B, NH, NW, device=dev, dtype=torch.uint8) for _ in range(nrot)]
    vis = [torch.empty_like(f) for f in frames]
    pal = torch.tensor(np.ascontiguousarray(np.asarray(O.ROAD_PALETTE)[:, ::-1]) * 255.0).round().to(torch.uint8).to(dev)   # BGR, 10 colours
    M = 256
    host = torch.empty(B * M * 44 + 4 * B, dtype=torch.uint8).pin_memory()
    g = np.random.default_rng(0)
    noise = g.integers(1, 10, (B, NH, NW), dtype=np.uint8)
    noise[g.random(noise.shape) >= 0.3] = 0
    noise = torch.from_numpy(noise).to(dev)

    def infer(i):
        k = i % nrot
        b200seg.preprocess_image(frames[k], target_size=(NW, NH), dtype=torch.bfloat16, out=xn[k], want_rgb=False)
        return model.predict_mask(xn[k], out=masks[k])

    def detect(mask):
        return b200seg.detect_objects(mask, CLASSES, size=(FW, FH), close=CLOSE, max_objects=M)

    def leg_b(i):
        det = detect(infer(i))
        host.copy_(det._buf, non_blocking=True)
        return det

    def leg_c(i):
        leg_b(i)
        k = i % nrot
        b200seg.overlay(frames[k], masks[k], pal, 0.7, 0.3, out=vis[k])

    legs = {
        "a_preprocess_predict_mask": infer,
        "b_plus_detect_objects_d2h": leg_b,
        "c_plus_overlay": leg_c,
        "d_detect_objects_alone": lambda i: detect(masks[i % nrot]),
        "e_detect_objects_noise": lambda i: detect(noise),
    }
    res = {"device": _device_info(dev), "batch": B, "frame": [FH, FW, 3], "network_input": [3, NH, NW], "classes": CLASSES,
           "close": CLOSE, "min_area": 0, "max_objects": M, "model": "MobileNetV2UNet(10), F2 weights, module .bfloat16(), eval",
           "steps": args.steps, "warmup": args.warmup, "legs": {}}
    with torch.no_grad():
        for k in range(nrot):
            infer(k)
        for name, fn in legs.items():
            sec = _time(fn, args.steps, args.warmup)
            res["legs"][name] = {"frames_per_s": round(B * args.steps / sec, 1), "us_per_batch": round(sec / args.steps * 1e6, 1)}

        # correctness on this run's data: detect_objects against the cv2 recipe for a subsample of frames
        infer(0)
        det = detect(masks[0])
        rows = det.to_list()
        counts = det.count.cpu().tolist()
        mask_np = masks[0].cpu().numpy()
        ref, cv_sec, cv_threads = _cv2_recipe(mask_np, args.cv2_frames)
        assert all(c <= M for c in counts), counts
        assert rows[:args.cv2_frames] == ref, "detect_objects differs from the cv2 recipe"
        res["objects_per_frame_mean"] = round(sum(counts) / B, 2)
        res["cv2_recipe"] = {"frames": args.cv2_frames, "ms_per_frame": round(cv_sec / args.cv2_frames * 1e3, 3),
                             "frames_per_s": round(args.cv2_frames / cv_sec, 1), "cv2_threads": cv_threads,
                             "host_cpus": os.cpu_count(), "rows_equal_detect_objects": True}
        ndet = detect(noise)
        res["noise_components_per_frame_mean"] = round(float(ndet.count.double().mean()), 1)

        # bytes from the shapes against the data-sheet bandwidth
        nb = _bytes(B, NH, NW, len(CLASSES), M)
        for name in ("d_detect_objects_alone", "e_detect_objects_noise"):
            us = res["legs"][name]["us_per_batch"]
            res["legs"][name].update({"bytes_model": int(nb), "TB_per_s": round(nb / us / 1e6, 3),
                                      "hbm_fraction": round(nb / (us * 1e-6) / HBM_BW, 4)})
        ob = B * FH * FW * 3 * 2 + B * NH * NW
        us = res["legs"]["c_plus_overlay"]["us_per_batch"] - res["legs"]["b_plus_detect_objects_d2h"]["us_per_batch"]
        res["overlay_increment"] = {"us_per_batch": round(us, 1), "bytes": int(ob), "hbm_fraction_of_increment": round(ob / (us * 1e-6) / HBM_BW, 3)
                                    if us > 0 else None}

        # kernel times of detect_objects (a separate profiler pass; not used for the rates above)
        from torch.profiler import ProfilerActivity, profile
        kern = {}
        for tag, mk in (("masks", masks[0]), ("noise", noise)):
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(10):
                    detect(mk)
                    b200seg.overlay(frames[0], masks[0], pal, 0.7, 0.3, out=vis[0])
                torch.cuda.synchronize()
            kern[tag] = {}
            for e in prof.key_averages():
                if any(s in e.key for s in ("close_init", "ccl_", "overlay_kernel")):
                    name = e.key.split("(")[0].replace("void ", "").replace("b200::", "")
                    t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
                    kern[tag][name] = round(float(t) / max(e.count, 1), 1)
        res["kernel_us_per_call"] = kern
    L = res["legs"]
    a = L["a_preprocess_predict_mask"]["us_per_batch"]
    res["detect_cost_vs_floor"] = round(L["b_plus_detect_objects_d2h"]["us_per_batch"] / a, 3)
    res["detect_vs_cv2_frames_per_s"] = round(L["d_detect_objects_alone"]["frames_per_s"] / res["cv2_recipe"]["frames_per_s"], 1)
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
