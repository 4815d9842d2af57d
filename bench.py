#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 segmentation hot path (BASELINE.json `metric`).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload infer|train] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

Default workload (N=1): BASELINE config[1] -- MobileNetV2UNet bf16 inference, batch 64 per GPU at
3x256x512, 10 classes, random-init weights, synthetic frames; frames are sharded across ranks with no
collective (weak scaling).  One "step" = one forward pass over one batch.

Every default run also times BASELINE config[2] -- the data-parallel training step (batch 32/GPU, bf16 activations, fused
Adam, bucketed all-reduce inside the backward graph when N > 1) -- for the same --steps/--warmup and reports it as numeric
`train_*` keys inside `config`, next to the torch-eager (cuDNN) incumbent on the same GPU (`eager_*` keys, N=1 only).

One JSON line on rank 0:
  value     images/s, whole job, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e       same metric through the public API with HOST (pinned) frames: H2D copy + forward +
            fused argmax mask + D2H of the mask inside the timed region (the inference.py:159-166 loop)
  roofline  the dominant kernel's achieved HBM GB/s (or TFLOP/s) vs MEASURED_PEAKS.json, measured
            live with CUDA events on the launch stream
  cpu_baseline  the oracle port of the reference path (fp32, PyTorch CPU) on this box's host cores
--impl reference: times that CPU path alone: the real reference (/root/reference via the Appendix-D shim) when that
tree is present, else its restatement oracle/unet_oracle.py (the GPU box has no /root/reference); `kind` says which ran.

--dump-outputs DIR: rank 0 writes what each timed leg returned in its last timed step as DIR/<name>.npy (float32):
logits (value leg), mask (e2e leg), train_loss and train_params (training leg: the loss and the weights the step updated).
Inputs and weights are seeded, so two builds run with the same arguments can be compared output for output.  The
inference arrays repeat bit for bit; the training ones only to rounding (BatchNorm sums depend on atomic order, and Adam's
normalised update magnifies that in weights whose gradients are near zero: measured on a B200 at 1000 W, two runs of the
default line differed by up to 5e-4 in train_loss and 4e-3 in train_params).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "team02-objectdetection_b200"))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

H, W, NCLS = 256, 512, 10


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="infer", choices=["infer", "train", "infer720", "unet_train"],
                    help="infer = BASELINE config[1] (default); train = config[2]; infer720 = config[4] (3x720x1280 padded to 736, "
                         "batch 8/GPU); unet_train = config[3] (plain UNet, 3x512x1024, bf16)")
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default 64 infer / 32 train)")
    ap.add_argument("--breakdown", action="store_true", help="print the per-kernel table to stderr")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train-leg", action="store_true", help="skip the config[2] training leg of the default run")
    ap.add_argument("--no-eager-baseline", action="store_true", help="skip the torch-eager incumbent legs (N=1)")
    ap.add_argument("--sustain-seconds", type=float, default=2.0, help="length of the extra sustained-throughput loop")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step of every leg to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the b200 path; --impl reference has no outputs to dump")
    return args


DUMP_ELEMS = 1 << 22        # float32 values per dumped array (16 MB): the four arrays stay under 64 MB at any batch
DUMP_SEED = 1234


def output_dumper(out_dir, rank):
    """dump(name, tensor) for --dump-outputs, or None.  A tensor of at most DUMP_ELEMS values is written whole; a larger
    one as the values at DUMP_ELEMS seeded positions of its flattened form (the same positions for the same shape, in
    ascending order), so that two runs with the same arguments write comparable arrays."""
    if not out_dir or rank != 0:
        return None
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)

    def dump(name, t):
        t = t.detach()
        if t.numel() > DUMP_ELEMS:
            g = torch.Generator().manual_seed(DUMP_SEED)
            idx = torch.randint(t.numel(), (DUMP_ELEMS,), generator=g).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())
    return dump


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm=d["hbm_gbs"], tc_burst=d["bf16_tflops"], tc=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tc_burst=1590.0, tc=1400.0, src="fallback")


E2E_TRACE = [] if os.environ.get("B200SEG_E2E_TRACE") else None     # debug: (host time, device event) after every e2e step
LEAD_IN = 4         # untimed steps queued ahead of the timed window (see the value leg)


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (B200_PROFILING.md's clocks line).

    Sampled in-process through NVML (pynvml: two light calls every 20 ms from a background thread).  The nvidia-smi CLI
    is only the fallback: measured on this pool, each of its queries stalls kernel submission for ~8 ms (and its first
    start on a fresh box for 25-30 ms), which inflated a 52 ms timed region from 2.62 to 3.0-4.3 ms/step."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index, self.first = [], None, index, 0
        self.nvml, self.handle, self.stop_flag, self.thread, self.max_mhz = None, None, False, None, None
        self.poll_log = []

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.thread.start()
            return
        except Exception:                                   # noqa: BLE001 -- no NVML binding: nvidia-smi CLI
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _poll_nvml(self):
        n = self.nvml
        names = (("hw_slowdown", n.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", n.nvmlClocksEventReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", n.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", n.nvmlClocksEventReasonSwPowerCap))
        while not self.stop_flag:
            try:
                _t = time.perf_counter()
                mhz = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                mask = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                self.poll_log.append((_t, time.perf_counter()))
                self.rows.append([str(mhz), str(self.max_mhz)] + [("Active" if mask & bit else "Not Active") for _, bit in names])
            except Exception:                               # noqa: BLE001
                pass
            time.sleep(0.02)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def mark(self):
        """Start of the timed region: only samples taken from here on are reported.  The sampler is started at process
        start and we WAIT here until it has delivered its first sample (the nvidia-smi fallback needs seconds on a fresh
        box)."""
        if self.nvml is not None or self.proc is not None:
            t0 = time.time()
            while not self.rows and time.time() - t0 < 20.0 and (self.nvml is not None or self.proc.poll() is None):
                time.sleep(0.05)
        self.first = len(self.rows)

    def stop(self):
        if self.nvml is None and self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        if self.nvml is not None:
            time.sleep(0.03)
            self.stop_flag = True
        else:
            time.sleep(0.15)
            self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in (self.rows[self.first:] or self.rows):
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def cpu_reference_leg(seconds=12.0, warmup=2, fixed_iters=None):
    """The reference's CPU path (fp32, batch 1 at 3x256x512, eval) on the host cores: see bench_baselines.cpu_leg."""
    from bench_baselines import cpu_leg
    return cpu_leg(seconds, warmup, fixed_iters)


_REAL_STDOUT = None


def protect_stdout():
    """stdout carries exactly ONE JSON line: libraries that write to fd 1 (NCCL's version banner under NCCL_DEBUG) are
    sent to stderr for the whole run and emit() writes the line to the original descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def shutdown(dist) -> None:
    """Leave the process group without ever hanging the launcher: NCCL's communicator teardown blocks while anything that
    captured its collectives is still alive, so it runs under a watchdog that ends the process (the JSON line is out)."""
    if dist is None:
        return
    t = threading.Timer(20.0, lambda: os._exit(0))
    t.daemon = True
    t.start()
    try:
        torch.cuda.synchronize()
        dist.destroy_process_group()
    finally:
        t.cancel()


def emit(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_REAL_STDOUT, data)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.perf_counter()
    per_step = max(1, 1)
    base = cpu_reference_leg(seconds=0, warmup=max(args.warmup, 1), fixed_iters=max(args.steps, 1) * per_step)
    wall = time.perf_counter() - t0
    line = {"impl": "reference", "metric": "MobileNetV2UNet inference images/s", "value": base["value"],
            "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": base["ms_per_image"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"MobileNetV2UNet eval forward, 3x{H}x{W}, {NCLS} classes, random init; CPU sample: "
                                   "batch 1 per step (reference inference.py is batch-1)", "device": "host CPU"},
            "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": base["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": wall}
    emit(line)


def main():
    args = parse()
    protect_stdout()
    if args.impl == "reference":
        return run_reference(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (B200); there is no CPU fallback for the product path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import b200seg
    from b200seg import _cabi
    sms, cc = _cabi.device_info()

    # nvidia-smi is started NOW, seconds before the timed region: its NVML initialisation stalls kernel launches for tens of
    # milliseconds on a fresh box (measured: a 54 ms timed region read 4.0-4.3 ms/step instead of 2.66 when it overlapped)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    dump = output_dumper(args.dump_outputs, rank)
    if args.workload in ("train", "unet_train"):
        from bench_train import run_train          # training step benchmark lives in its own file
        return run_train(args, dev, dist, world, rank, peaks(), clocks, emit, shutdown, dump)

    global H, W
    if args.workload == "infer720":
        H, W = 736, 1280                            # 720 rows padded to a multiple of 32 (the reference fails on 720, SURVEY finding 8)
    B = args.batch or (8 if args.workload == "infer720" else 64)
    torch.manual_seed(0)
    model = b200seg.MobileNetV2UNet(output_channels=NCLS).to(dev).bfloat16().eval()
    eng = model._get_engine()
    g = torch.Generator(device="cpu").manual_seed(rank)
    nrot = 4                                           # rotating inputs; activations (~7 GB/step) >> 126 MB L2 anyway
    xs = [torch.randn(B, 3, H, W, generator=g).bfloat16().to(dev) for _ in range(nrot)]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- value leg: inputs resident in HBM ----------------
    settle = 30        # extra untimed steps after the W warm-up steps: the first ~10 replays after capture run 3-5 % slow
    with torch.no_grad():
        y = None
        for i in range(args.warmup + settle):
            # bound to a name exactly like the timed loop: the loop then needs TWO output blocks alive at a time (the new
            # result is allocated before the old one is released); a warm-up that drops its result keeps only one in the
            # caching allocator and the second timed step pays a 168 MB cudaMalloc (20-160 ms, host AND device stalled)
            y = model(xs[i % nrot])
        barrier()
        clocks.mark()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        # lead-in: a few untimed steps are queued first so that the host is several steps ahead of the device when the
        # timed window opens -- the 20-step window is ~40 ms of device time, and a single host-side submission stall (the
        # clock sampler's NVML query holds a driver lock for milliseconds now and then) otherwise shows up as a 30 %
        # slower "step".  The events still bracket EXACTLY args.steps steps, executed back to back on the device.
        for i in range(LEAD_IN):
            y = model(xs[i % nrot])
        e0.record()
        vtrace = []
        for i in range(args.steps):
            y = model(xs[(i + LEAD_IN) % nrot])
            if E2E_TRACE is not None:
                ev = torch.cuda.Event(enable_timing=True); ev.record()
                vtrace.append((time.perf_counter(), ev))
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if vtrace and rank == 0:
            h0 = vtrace[0][0]
            print("value trace (step: host issue ms, device done ms): " +
                  " ".join(f"{i}:{(h - h0) * 1e3:.1f}/{e0.elapsed_time(d):.1f}" for i, (h, d) in enumerate(vtrace)), file=sys.stderr)
            print("sampler polls (start ms, duration ms): " + " ".join(f"{(a - h0) * 1e3:.1f}/{(b - a) * 1e3:.2f}" for a, b in clocks.poll_log[-12:]),
                  file=sys.stderr)
        clk = clocks.stop() if rank == 0 else None
        if dump is not None:
            dump("logits", y)                       # y: the last timed step's result
        # sustained figure: the same loop for >= --sustain-seconds (power/thermals settled), reported beside `value`
        n_sus = max(args.steps, int(args.sustain_seconds * 1e3 / max(ms / args.steps, 1e-3)))
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for i in range(n_sus):
            y = model(xs[i % nrot])
        s1.record()
        torch.cuda.synchronize()
        ms_sus = s0.elapsed_time(s1) / n_sus

    # ---------------- e2e leg: host frames in, class mask out ----------------
    # the reference's per-frame flow (inference.py:28-46,162-164): uint8 BGR camera frame -> preprocess_image -> model ->
    # argmax.  Frames arrive at the network size (the resize path is exercised by the tests); only uint8 crosses PCIe.
    xh = [torch.randint(0, 256, (B, H, W, 3), generator=g, dtype=torch.uint8).pin_memory() for _ in range(2)]
    mh = [torch.empty(B, H, W, dtype=torch.uint8).pin_memory() for _ in range(2)]
    xd = [torch.empty(B, H, W, 3, dtype=torch.uint8, device=dev) for _ in range(2)]
    xn = [torch.empty(B, 3, H, W, dtype=torch.bfloat16, device=dev) for _ in range(2)]
    md = [torch.empty(B, H, W, dtype=torch.uint8, device=dev) for _ in range(2)]      # device masks, double-buffered: no
    # per-frame allocation (a fresh mask handed to the download stream with record_stream() cannot be recycled until its
    # event completes; with the host several frames ahead the caching allocator fell back to cudaMalloc/cudaFree -- a
    # device-wide sync of 20-170 ms in the middle of the timed window)
    copy_s, out_s, comp_s = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.current_stream()
    own_d2h = os.environ.get("B200SEG_E2E_D2H_STREAM", "1") != "0"

    def e2e_steps(n, lead=0, t_start=None):
        # double-buffered: H2D of step i+1 overlaps the forward of step i; every copy is inside the timed region.
        # ``lead`` untimed steps run first in the same pipeline (see LEAD_IN): the window opens on the compute stream in
        # steady state, so the H2D of a timed step overlaps the step before it and the D2H of the last lead-in step falls
        # inside the window -- n uploads, n forwards and n downloads are timed.
        ev_in = [torch.cuda.Event() for _ in range(2)]
        ev_free = [torch.cuda.Event() for _ in range(2)]
        ev_out = [torch.cuda.Event() for _ in range(2)]
        for i in range(lead + n):
            k = i & 1
            if i == lead and t_start is not None:
                t_start.record()
            with torch.cuda.stream(copy_s):
                if i >= 2:
                    copy_s.wait_event(ev_free[k])
                xd[k].copy_(xh[k], non_blocking=True)
                ev_in[k].record(copy_s)
            comp_s.wait_event(ev_in[k])
            b200seg.preprocess_image(xd[k], target_size=(W, H), dtype=torch.bfloat16, out=xn[k], want_rgb=False)
            if i >= 2:
                comp_s.wait_event(ev_out[k])             # the download of frame i-2 has left md[k]
            mask = model.predict_mask(xn[k], out=md[k])
            ev_free[k].record(comp_s)
            if E2E_TRACE is not None:
                ev = torch.cuda.Event(enable_timing=True); ev.record(comp_s)
                E2E_TRACE.append((time.perf_counter(), ev))
            if own_d2h:
                with torch.cuda.stream(out_s):           # the D2H of the mask overlaps the next forward as well (own stream:
                    out_s.wait_event(ev_free[k])         # on the H2D stream it would hold back the next frame upload)
                    mh[k].copy_(mask, non_blocking=True)
                    ev_out[k].record(out_s)
            else:
                mh[k].copy_(mask, non_blocking=True)
                ev_out[k].record(comp_s)
        torch.cuda.synchronize()

    with torch.no_grad():
        e2e_steps(max(12, args.warmup))         # untimed: first touches of the pinned buffers / copy engines on a fresh box
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if E2E_TRACE is not None:
            E2E_TRACE.clear()
        e2e_steps(args.steps, LEAD_IN, t0)
        t1.record()
        barrier()
        ms_e2e = t0.elapsed_time(t1)
        if dump is not None:
            dump("mask", mh[(LEAD_IN + args.steps - 1) & 1])      # the host mask of the last timed step
        if E2E_TRACE is not None and rank == 0:
            h0, d0 = E2E_TRACE[0]
            print("e2e trace (step: host issue ms, device done ms): " +
                  " ".join(f"{i}:{(h - h0) * 1e3:.1f}/{d0.elapsed_time(d):.1f}" for i, (h, d) in enumerate(E2E_TRACE)), file=sys.stderr)

    # ---------------- per-kernel roofline (live, CUDA events on the launch stream) ----------------
    pk = peaks()
    acc = {}
    with torch.no_grad():
        for it in range(3 + 5):
            prof, penv = [], {}
            ppk = eng._pack_eval(eng._mode(xs[0]))
            eng.forward_eval(xs[it % nrot], profile=prof, keep=penv)
            torch.cuda.synchronize()
            if it < 3:
                continue
            for s, a, b, nbytes, flops in prof:
                r = acc.setdefault(s.name, dict(op=s.op, taps=s.taps, ms=0.0, bytes=nbytes, flops=flops, n=0,
                                                lbytes=eng.layer_model_bytes(s, penv, ppk),
                                                shape=(tuple(s.conv.weight.shape) if s.op == "dense" else None)))
                r["ms"] += a.elapsed_time(b); r["n"] += 1
    FUSED = ("mbconv", "stem_mb1", "tail")
    rows = []
    for name, r in acc.items():
        t = r["ms"] / r["n"] * 1e-3
        # HBM figure per SURVEY 8(d)'s per-LAYER traffic model (lbytes: a fused kernel is credited with the layers it replaces);
        # gbs_io = the same on the kernel's own input + output bytes.  Unfused kernels: identical.
        gbs, gbs_io, tfs = r["lbytes"] / t / 1e9, r["bytes"] / t / 1e9, r["flops"] / t / 1e12
        bound = "tensor" if (r["flops"] / max(r["lbytes"], 1)) > pk["tc"] * 1e3 / pk["hbm"] else "hbm"
        rows.append(dict(name=name, op=r["op"], us=t * 1e6, gbs=gbs, gbs_io=gbs_io, tfs=tfs, bound=bound, bytes=r["bytes"],
                         lbytes=r["lbytes"], flops=r["flops"], shape=r["shape"], taps=r["taps"],
                         frac=(tfs / pk["tc_burst"]) if bound == "tensor" else gbs / pk["hbm"]))
    rows.sort(key=lambda r: -r["us"])
    tot_us = sum(r["us"] for r in rows)
    if args.breakdown and rank == 0:
        print(f"{'kernel':34s} {'op':8s} {'us':>9s} {'share':>6s} {'GB/s':>8s} {'io GB/s':>8s} {'TF/s':>8s} bound  frac", file=sys.stderr)
        for r in rows:
            print(f"{r['name']:34s} {r['op']:8s} {r['us']:9.1f} {r['us'] / tot_us:6.1%} {r['gbs']:8.0f} {r['gbs_io']:8.0f} {r['tfs']:8.1f} "
                  f"{r['bound']:6s} {r['frac']:.2f}", file=sys.stderr)
        print(f"sum of kernels {tot_us:.0f} us; step {ms / args.steps * 1e3:.0f} us   (GB/s: SURVEY 8d per-layer traffic model -- fused kernels "
              f"are credited with the layers they replace; io GB/s: the kernel's own input + output bytes)", file=sys.stderr)
    top = rows[0]
    roofline = {"kernel": top["name"], "bound": top["bound"],
                "achieved": top["tfs"] if top["bound"] == "tensor" else top["gbs"],
                "peak": pk["tc_burst"] if top["bound"] == "tensor" else pk["hbm"],
                "unit": "TFLOP/s" if top["bound"] == "tensor" else "GB/s", "frac": top["frac"], "traffic": None,
                "peak_source": pk["src"], "share_of_step": top["us"] / tot_us,
                "algorithmic_per_launch": top["flops"] if top["bound"] == "tensor" else top["lbytes"]}
    if top["op"] in FUSED:
        roofline["fused_io_bytes_per_launch"] = top["bytes"]
        roofline["frac_on_fused_io_bytes"] = top["gbs_io"] / pk["hbm"]
        roofline["note"] = ("fused kernel: algorithmic bytes = SURVEY 8(d) per-layer model summed over the layers it replaces (their "
                            "intermediates stay on chip, see traffic); its own bound is CUDA-core issue, DESIGN.md section 4")
    if top.get("shape"):
        # third bound of a small-N implicit GEMM: the tcgen05.mma issue floor measured by tools/mma_probe.py
        # (profiles/r01_mma_probe.txt): cycles per M=128, K=16 instruction as a function of N, per SM
        cout, cin, taps = top["shape"][0], top["shape"][1], top["taps"]
        n_tile = min((cout + 15) // 16 * 16, 256)
        table = [(16, 39.0), (32, 40.0), (64, 48.0), (128, 64.0), (256, 128.0)]
        cyc = next(c for n, c in table if n_tile <= n)
        ksteps = sum((min(64, cin - c0) + 15) // 16 for c0 in range(0, cin, 64))
        pixels = top["flops"] / (2.0 * cout * taps * cin)
        n_mma = (pixels / 128.0) * taps * ksteps * ((cout + n_tile - 1) // n_tile)
        floor_us = n_mma * cyc / sms / ((clk or {}).get("sm_mhz") or 1965.0)
        roofline["mma_issue_floor_us"] = floor_us
        roofline["frac_of_mma_issue_floor"] = floor_us / top["us"]
        roofline["note"] = ("small-N implicit GEMM: bound by the tcgen05.mma issue floor (cycles per instruction do not shrink "
                            "below ~40 for N < 96), not by HBM; see DESIGN.md finding 8")
    try:                                   # DRAM traffic of the dominant kernel from the committed ncu capture, if it is the same kernel
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            ent = json.load(f).get(top["name"])
        if ent and B == 64 and args.workload == "infer":
            roofline["traffic"] = ent["traffic_bytes"]
            roofline["traffic_source"] = ent["capture"]
    except (OSError, ValueError):
        pass
    tot_bytes = sum(r["bytes"] for r in rows)
    tot_lbytes = sum(r["lbytes"] for r in rows)      # = SURVEY 8d's 115.7 MB/img x B for the MobileNetV2UNet inference step
    step_s = ms / args.steps * 1e-3
    step_roofline = {"bound": "hbm", "algorithmic_bytes_per_step": tot_lbytes,
                     "note": "SURVEY 8(d) per-layer traffic model (the 115.7 MB/img figure); fused_io_*: bytes the schedule actually "
                             "has to move (fused blocks count input + output only)",
                     "achieved": tot_lbytes / step_s / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                     "frac": tot_lbytes / step_s / 1e9 / pk["hbm"],
                     "fused_io_bytes_per_step": tot_bytes, "frac_on_fused_io_bytes": tot_bytes / step_s / 1e9 / pk["hbm"]}

    # ---------------- max over ranks ----------------
    if dist is not None:
        t = torch.tensor([ms, ms_e2e, ms_sus], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e, ms_sus = float(t[0]), float(t[1]), float(t[2])

    # ---------------- config[2]: the training step (every rank; data parallel when N > 1) ----------------
    train = None
    if args.workload == "infer" and not args.no_train_leg:
        del xs, xd, xn, y
        eng._graphs.clear()
        torch.cuda.empty_cache()
        from bench_train import train_leg
        train = train_leg(args, dev, dist, world, rank, dump=dump)
    if rank != 0:
        shutdown(dist)
        return
    eager = {}
    if world == 1 and args.workload == "infer" and not args.no_eager_baseline:
        from bench_baselines import gpu_eager_leg
        eager = gpu_eager_leg(dev)

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference_leg()
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
    n_launch = len(eng._schedule("bf16", "tc", H, W))      # kernels per forward (fused inverted-residual blocks count once)
    line = {"metric": "MobileNetV2UNet inference images/s", "value": B * world * args.steps / (ms * 1e-3),
            "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"MobileNetV2UNet bf16 inference, batch {B}/GPU, 3x{H}x{W}, {NCLS} classes, random init "
                                   + ("(BASELINE config[4]: 720x1280 frames padded to 736 rows; " if args.workload == "infer720" else "(BASELINE config[1]; ")
                                   + "frames sharded by rank, no collective)",
                       "global_batch": B * world, "l2": "4 rotating input batches; ~7 GB of activations per step >> 126 MB L2",
                       "sm_count": sms, "cc": cc, "settle_steps_untimed": settle, "sustained_img_s": B * world / (ms_sus * 1e-3), "sustained_steps": n_sus},
            "e2e": {"value": B * world * args.steps / (ms_e2e * 1e-3), "unit": "images/s",
                    "h2d_bytes_per_step": B * 3 * H * W, "d2h_bytes_per_step": B * H * W,
                    "api": "b200seg.preprocess_image(uint8 BGR HWC frames, pinned) -> model.predict_mask(...) -> uint8 class mask "
                           "(inference.py:28-46,162-164 on the GPU: bit-exact resize/normalise, fused final upsample + argmax), "
                           "double-buffered copies"},
            "gpu_launches": n_launch * args.steps, "launches_per_step": n_launch,
            "roofline": roofline, "step_roofline": step_roofline, "clocks": clk}
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if train is not None:
        # BASELINE config[2], numeric keys only (train.py:31-42 loop body; see bench_train.py): whole-job images/s
        line["config"].update({
            "train_img_s": train["img_s"], "train_ms_per_step": train["ms_per_step"], "train_e2e_img_s": train["e2e_img_s"],
            "train_roofline_frac": train["achieved_gbs"] / pk["hbm"], "train_batch_per_gpu": train["B"],
            "train_host_issue_ms": train["host_issue_ms_per_step"], "allreduce_exposed_ms": train["allreduce_exposed_ms"],
            "train_launches_per_step": train["launches_per_step"], "train_last_loss": train["last_loss"]})
    for k, v in eager.items():
        line["config"][k] = v
    emit(line)
    shutdown(dist)


if __name__ == "__main__":
    main()
