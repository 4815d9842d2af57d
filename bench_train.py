"""Training-step benchmark (BASELINE config[2]): MobileNetV2UNet fwd + pixel CE + bwd + Adam, batch 32 per GPU at
3x256x512, data parallel over the ranks.  `train_leg()` is run by EVERY default `python bench.py --gpus N` (its numbers are
the `train_*` keys of the line's `config`), and `python bench.py --workload train` prints it as the headline instead.

A step is exactly the reference's loop body (train.py:35-39): optimizer.zero_grad(); outputs = model(inputs);
loss = criterion(outputs, targets); loss.backward(); optimizer.step() -- with Adam(lr=1.5e-4) (main.py:100) and, for N>1,
the bucketed gradient all-reduce of b200seg.dp overlapped with backward inside the captured backward graph.
"""
import os
import sys
import time

import torch

NCLS = 10
TRAIN_BYTES_PER_IMG = 353e6        # SURVEY 8d: MobileNetV2UNet train, bf16 activations, 3x256x512
UNET_BYTES_PER_IMG = 4772e6        # SURVEY 8d: UNet(10) train, bf16 activations, 3x512x1024


def train_leg(args, dev, dist, world, rank, unet=False, batch=0, want_breakdown=False, clocks=None, dump=None):
    """Times the training step three ways (device-resident inputs; end to end from pinned host batches with loss.item()
    every step; for N>1 the same step with the collectives detached = the exposed all-reduce time).  Returns a dict of
    plain numbers (max over ranks where it matters) + the per-layer trace of one warm eager step.  ``dump`` (bench.py's
    --dump-outputs) receives the loss and the weights of the last device-resident timed step."""
    import b200seg
    from b200seg import dp, train_path
    H, W = (512, 1024) if unet else (256, 512)
    B = batch or (4 if unet else 32)
    precision = os.environ.get("B200SEG_TRAIN_PRECISION", "bf16")     # bf16 activations + tcgen05 convs, fp32 master weights
    fused_adam = os.environ.get("B200SEG_BENCH_ADAM", "fused") == "fused"
    torch.manual_seed(0)
    model = (b200seg.UNet(output_channels=NCLS) if unet else b200seg.MobileNetV2UNet(output_channels=NCLS)).to(dev)
    eng = model._get_engine()
    eng.precision = precision
    if dist is not None:
        dp.broadcast_model(model)
        dp.attach(model)
    criterion = b200seg.CrossEntropyLoss()
    # main.py:100 -- same constructor call; b200seg.Adam is the one-launch multi-tensor drop-in for optim.Adam
    optimizer = (b200seg.Adam if fused_adam else torch.optim.Adam)(model.parameters(), lr=1.5e-4)
    model.train()
    g = torch.Generator(device="cpu").manual_seed(rank)
    nrot = 2
    xs = [torch.randn(B, 3, H, W, generator=g).to(dev) for _ in range(nrot)]
    ys = [torch.randint(0, NCLS, (B, H, W), generator=g).to(dev) for _ in range(nrot)]

    def step(x, y):
        optimizer.zero_grad()
        out = model(x)
        loss = criterion(out, y)
        loss.backward()
        optimizer.step()
        return loss

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(n):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        th0 = time.perf_counter()
        for i in range(n):
            loss = step(xs[i % nrot], ys[i % nrot])
        host = (time.perf_counter() - th0) * 1e3 / n          # host time to ISSUE a step (no sync inside)
        e1.record()
        barrier()
        return e0.elapsed_time(e1), host, loss

    for i in range(max(args.warmup, eng.graph_after + 2)):    # eager steps, graph capture, first replays
        step(xs[i % nrot], ys[i % nrot])
    barrier()
    if clocks is not None:
        clocks.mark()
    from b200seg._cabi import LAUNCHES
    n0 = LAUNCHES[0]
    ms, host_issue_ms, loss = timed(args.steps)
    in_graph = max([e["graph"].n_launches for e in eng._graphs.values() if e.get("graph") is not None and hasattr(e["graph"], "n_launches")] or [0])
    launches_per_step = in_graph + (LAUNCHES[0] - n0) / args.steps      # kernels replayed from the two graphs + launched directly
    clk = clocks.stop() if (clocks is not None and rank == 0) else None
    last_loss = float(loss)
    if dump is not None:
        dump("train_loss", loss)
        dump("train_params", torch.cat([p.detach().reshape(-1) for p in model.parameters()]))

    # e2e: host (pinned) fp32 images + int64 labels in, loss.item() out, every step.  Input feed (SURVEY 8f rank 4):
    # non-blocking uploads on a copy stream, one batch ahead -- the upload of batch i+1 overlaps step i although the loss is
    # read back (a sync) every step as train.py:41-42 does
    xh = [torch.randn(B, 3, H, W, generator=g).pin_memory() for _ in range(2)]
    yh = [torch.randint(0, NCLS, (B, H, W), generator=g).pin_memory() for _ in range(2)]

    # the library input feed (b200seg.DeviceFeeder, SURVEY 8f rank 4) in place of train.py:32-33's blocking copies; one
    # feeder for the whole leg (its device buffers are allocated on the untimed first pass)
    feeder = b200seg.DeviceFeeder([], dev)

    def e2e_steps(n):
        feeder.loader = [(xh[i & 1], yh[i & 1]) for i in range(n)]
        for x, y in feeder:
            step(x, y).item()                       # train.py:41-42 reads the loss every step

    e2e_steps(3)
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    e2e_steps(args.steps)
    t1.record()
    barrier()
    ms_e2e = t0.elapsed_time(t1)

    # exposed all-reduce time: the same step with the collectives detached (every rank still steps; replicas drift apart,
    # which no longer matters -- this is the last thing the leg does with the model)
    ms_nocomm = None
    if dist is not None:
        del loss
        dp.detach(model)                     # also releases the graphs that captured NCCL collectives
        for i in range(eng.graph_after + 3):
            step(xs[i % nrot], ys[i % nrot])
        ms_nocomm, _, _ = timed(args.steps)

    # per-layer forward/backward times of one WARM eager step (CUDA events on the launch stream): the first traced step
    # pays the caching allocator's first-touch of the eager buffers (the graphs own their pool) and is discarded
    rows, tot = [], 0.0
    if want_breakdown:
        for rep in range(2):
            train_path.TRACE = []
            step(xs[0], ys[0])
            torch.cuda.synchronize()
            tr, train_path.TRACE = train_path.TRACE, None
        agg = {}
        for phase, name, a, b in tr:
            agg[(phase, name)] = agg.get((phase, name), 0.0) + a.elapsed_time(b)
        rows = sorted(agg.items(), key=lambda kv: -kv[1])
        tot = sum(v for _, v in rows)

    if dist is not None:
        t = torch.tensor([ms, ms_e2e, ms_nocomm, host_issue_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e, ms_nocomm, host_issue_ms = (float(v) for v in t)
    bytes_img = (UNET_BYTES_PER_IMG if unet else TRAIN_BYTES_PER_IMG) * (1 if precision == "bf16" else 2)
    step_s = ms / args.steps * 1e-3
    res = dict(B=B, H=H, W=W, precision=precision, fused_adam=fused_adam, ms_per_step=ms / args.steps,
               img_s=B * world / step_s, e2e_img_s=B * world * args.steps / (ms_e2e * 1e-3),
               host_issue_ms_per_step=host_issue_ms, last_loss=last_loss, bytes_per_step=bytes_img * B,
               achieved_gbs=bytes_img * B / step_s / 1e9,
               allreduce_exposed_ms=(ms - ms_nocomm) / args.steps if ms_nocomm is not None else 0.0,
               h2d_bytes_per_step=B * 3 * H * W * 4 + B * H * W * 8, rows=rows, rows_total=tot, clocks=clk,
               launches_per_step=launches_per_step)
    eng._graphs.clear()
    eng._train_ws = None
    del model, optimizer, xs, ys, feeder, eng
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    return res


def run_train(args, dev, dist, world, rank, pk, clocks, emit, shutdown, dump=None):
    unet = args.workload == "unet_train"
    r = train_leg(args, dev, dist, world, rank, unet=unet, batch=args.batch, want_breakdown=True, clocks=clocks, dump=dump)
    rows, tot = r["rows"], r["rows_total"]
    if args.breakdown and rank == 0:
        print(f"{'phase':4s} {'layer':34s} {'ms':>9s} {'share':>6s}", file=sys.stderr)
        for (phase, name), v in rows[:30]:
            print(f"{phase:4s} {name:34s} {v:9.3f} {v / tot:6.1%}", file=sys.stderr)
        print(f"sum fwd {sum(v for (p, _), v in rows if p == 'fwd'):.2f} ms, bwd {sum(v for (p, _), v in rows if p == 'bwd'):.2f} ms "
              f"(one warm eager step); graphed step {r['ms_per_step']:.2f} ms", file=sys.stderr)
    if rank != 0:
        shutdown(dist)
        return
    (top_phase, top_name), top_ms = rows[0]
    B, H, W = r["B"], r["H"], r["W"]
    name = "UNet" if unet else "MobileNetV2UNet"
    line = {"metric": name + " training images/s", "value": r["img_s"], "unit": "images/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if r["precision"] == "bf16" else "f32", "data": "synthetic",
            "config": {"workload": f"{name} training step (fwd + pixel CE + bwd + Adam), batch {B}/GPU, 3x{H}x{W}, {NCLS} classes "
                                   f"(BASELINE config[{3 if unet else 2}]); activations {r['precision']}, fp32 master weights, "
                                   f"{'b200seg.Adam (fused multi-tensor)' if r['fused_adam'] else 'torch.optim.Adam'}(lr=1.5e-4); "
                                   f"data parallel, per-replica BatchNorm, bucketed all-reduce inside the backward graph",
                       "global_batch": B * world, "l2": "~20 GB of activations per step >> 126 MB L2", "last_loss": r["last_loss"],
                       "host_issue_ms_per_step": r["host_issue_ms_per_step"], "allreduce_exposed_ms": r["allreduce_exposed_ms"]},
            "e2e": {"value": r["e2e_img_s"], "unit": "images/s",
                    "h2d_bytes_per_step": r["h2d_bytes_per_step"], "d2h_bytes_per_step": 4,
                    "api": "train.py:32-42 loop body: pinned fp32 images + int64 labels uploaded one batch ahead on a copy stream, step, loss.item() every step"},
            "roofline": {"kernel": f"whole step (top layer of a warm eager step: {top_phase}:{top_name})",
                         "bound": "hbm", "achieved": r["achieved_gbs"], "peak": pk["hbm"], "unit": "GB/s",
                         "frac": r["achieved_gbs"] / pk["hbm"], "traffic": None, "peak_source": pk["src"],
                         "note": "whole-step algorithmic bytes (SURVEY 8d model) / step time; per-layer shares in --breakdown",
                         "share_of_step": top_ms / tot},
            "gpu_launches": int(r["launches_per_step"] * args.steps), "launches_per_step": r["launches_per_step"], "clocks": r["clocks"]}
    emit(line)                # bench.py's emitter: the ONE stdout line (bench.py runs as __main__, do not re-import it)
    shutdown(dist)
