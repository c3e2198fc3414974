"""bench.py --workload train: the CVM_VIGOR training step (BASELINE.json configs[4]; reference train_VIGOR.py:96-157).

A step = forward (PyTorch encoders in train mode + the CUDA post-encoder path) + the reference's loss combination
(InfoNCE x6 + cross entropy + orientation loss, fused CUDA kernels) + backward (this library's backward kernels + PyTorch
autograd through the encoders) + bucketed NCCL gradient all-reduce overlapped with the backward + Adam(1e-4) step, on a
per-GPU batch of 8 synthetic pairs (the reference's default batch size, train_VIGOR.py:30) with synthetic ground truth of the
reference's statistics (datasets.py:142-166).  One process per GPU; weak scaling (every rank its own 8 pairs).

Same JSON contract as the inference workloads; extra key `allreduce` = {bytes, buckets, alone_ms, exposed_ms, overlap}.
"""
from __future__ import annotations

import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))

METRIC = "VIGOR training pairs/sec (CVM_VIGOR forward + losses + backward + gradient all-reduce + Adam step)"
DESC = ("CVM_VIGOR training step, synthetic VIGOR shape (3x320x640 + 3x512x512), InfoNCE + heatmap + orientation losses, "
        "DDP gradient all-reduce over NCCL, Adam lr 1e-4 (BASELINE.json configs[4])")
GROUND = (320, 640)


def _synthetic_batch(B, seed):
    from ccvpe_b200.synthetic import synthetic_ground_truth, synthetic_pair
    grd, sat = synthetic_pair(B, GROUND, seed=seed)
    gt, gt_with_ori, gt_orientation = synthetic_ground_truth(B, seed=seed)
    return [grd, sat, gt, gt_with_ori, gt_orientation]


def cpu_train_baseline(budget_s=60.0):
    """The reference's training step (oracle port of the forward + reference losses through torch autograd + Adam) on the
    host cores, batch 1, bounded."""
    from ccvpe_b200 import models
    from ccvpe_b200.synthetic import fill_deterministic
    from oracle import ccvpe_oracle as orc

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    model = models.CVM_VIGOR("cpu", True).train()
    fill_deterministic(model.state_dict(), seed=0)
    for n, p in model.named_parameters():
        p.requires_grad_("._fc." not in n)
    params = dict(model.named_parameters())
    opt = torch.optim.Adam([p for p in model.parameters() if p.requires_grad], lr=1e-4, betas=(0.9, 0.999))
    grd, sat, gt, gwo, gor = _synthetic_batch(1, 0)
    times = []
    t_begin = time.time()
    for i in range(4):
        t0 = time.time()
        opt.zero_grad()
        out = orc.forward_full("vigor", params, model.grd_efficientnet, model.sat_efficientnet, grd, sat)
        loss = orc.training_loss(out, gt, gwo, gor)
        loss.backward()
        opt.step()
        if i > 0:
            times.append(time.time() - t0)
        if time.time() - t_begin > budget_s and times:
            break
    best = min(times)
    return dict(value=1.0 / best, unit="pairs/s", cores=cores, kind="port",
                sample="oracle port of the CVM_VIGOR training step (forward + reference losses + torch autograd backward + Adam), "
                       "fp32, batch 1, best of %d after 1 warm-up (%.2f s/step, torch threads=%d)" % (len(times), best, cores))


def run_reference_arm(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    base = cpu_train_baseline(budget_s=120.0)
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": "pairs/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 / base["value"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": DESC + " -- CPU arm: bounded sample of batch 1 per step", "workload_key": "train",
                       "batch_per_gpu": args.batch or 8, "parallelism": "cpu"},
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main(args):
    if args.impl == "reference":
        return run_reference_arm(args)
    import bench as B_
    from ccvpe_b200 import cabi, losses, models
    from ccvpe_b200.ddp import GradientAllReducer
    from ccvpe_b200.decoder import OpTimer
    from ccvpe_b200.synthetic import fill_deterministic

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    Bsz = args.batch or 8
    model = models.CVM_VIGOR("cuda", True)
    fill_deterministic(model.state_dict(), seed=0)          # identical replicas on every rank
    model = model.to(dev).set_precision(args.precision).train()
    # PyTorch-side tuning of the (PyTorch) encoders: cuDNN autotuning, and channels-last inputs (below)
    torch.backends.cudnn.benchmark = True
    if args.backend == "simt":
        model.set_backend(cabi.BACKEND_SIMT)
    reducer = GradientAllReducer(model)
    use_graph = not args.no_cuda_graph
    opt = torch.optim.Adam([p for p in model.parameters() if p.requires_grad], lr=1e-4, betas=(0.9, 0.999), fused=True,
                           capturable=use_graph)
    host = [t.pin_memory() for t in _synthetic_batch(Bsz, 200 + rank)]
    resident = [t.to(dev) for t in host]
    # the model feeds its bf16-autocast encoders channels-last inputs: resident channels-last buffers make that conversion free
    resident[0] = resident[0].contiguous(memory_format=torch.channels_last)
    resident[1] = resident[1].contiguous(memory_format=torch.channels_last)

    def eager_step(grd, sat, gt, gwo, gor):
        reducer.zero_grad()
        out = model(grd, sat)
        loss = losses.training_loss(out, gt, gwo, gor)
        loss.backward()
        reducer.finish()
        opt.step()
        return loss.detach()

    graphed = [None]
    graph_note = None

    def step(batch):
        if graphed[0] is not None and model.pipeline.timer is None:
            return graphed[0](*batch)
        return eager_step(*batch)

    copy_stream = torch.cuda.Stream(device=dev)
    dev_in = [[torch.empty_like(t) for t in resident] for _ in range(2)]
    slot_free = [None, None]

    def upload(slot):
        with torch.cuda.stream(copy_stream):
            if slot_free[slot] is not None:
                copy_stream.wait_event(slot_free[slot])
            for d, h in zip(dev_in[slot], host):
                d.copy_(h, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return ev

    loss_host = torch.empty((), dtype=torch.float32).pin_memory()

    def run_e2e(steps):
        nxt = upload(0)
        last = None
        for i in range(steps):
            slot = i % 2
            ev = nxt
            if i + 1 < steps:
                nxt = upload(1 - slot)
            torch.cuda.current_stream().wait_event(ev)
            loss = step(dev_in[slot])
            slot_free[slot] = torch.cuda.Event()
            slot_free[slot].record()
            loss_host.copy_(loss.detach(), non_blocking=True)        # D2H of the step's result (the loss)
            done = torch.cuda.Event()
            done.record()
            done.synchronize()
            last = float(loss_host)
        return last

    sampler = B_.ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(2):
        step(resident)
    if use_graph:
        # the whole step as ONE CUDA graph (training.GraphedTrainStep); capture is an optimisation, never a requirement
        from ccvpe_b200.training import GraphedTrainStep
        try:
            graphed[0] = GraphedTrainStep(eager_step, resident, warmup=2)
            resident = graphed[0].static_in                     # the resident leg feeds the graph's own input buffers
            step(resident)
            torch.cuda.synchronize()
        except Exception as exc:                                # noqa: BLE001
            graphed[0] = None
            use_graph = False
            graph_note = "CUDA-graph capture of the training step failed (%s: %s); ran eagerly" % (type(exc).__name__, exc)
            torch.cuda.synchronize()
    for _ in range(max(args.warmup, 3)):
        step(resident)
    barrier()
    # ---- timed region: device-resident inputs ----
    cabi.reset_launch_count()
    barrier()
    w0 = time.time()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ncu_range = bool(os.environ.get("CCVPE_NCU_RANGE"))       # `ncu --profile-from-start off`: capture exactly these steps
    if ncu_range:
        torch.cuda.profiler.start()
    ev0.record()
    for _ in range(args.steps):
        loss = step(resident)
    ev1.record()
    if ncu_range:
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
    barrier()
    sampler.window(w0, time.time())
    launches = cabi.launch_count()
    ms_total = ev0.elapsed_time(ev1)
    final_loss = float(loss)
    # ---- per-kernel attribution: same steps with per-launch events ----
    timer = OpTimer()
    model.pipeline.timer = timer
    for _ in range(args.steps):
        step(resident)
    torch.cuda.synchronize()
    layers = timer.summary()
    model.pipeline.timer = None
    # ---- all-reduce: alone vs exposed ----
    ar = {"bytes": int(reducer.n_params) * 4, "buckets": reducer.bucket_bytes, "world": world}
    if world > 1:
        for _ in range(2):                          # (first eager collectives of these sizes: protocol / channel set-up)
            reducer.all_reduce_alone()
        barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(5):
            reducer.all_reduce_alone()
        a1.record()
        torch.cuda.synchronize()
        ar["alone_ms"] = round(a0.elapsed_time(a1) / 5, 3)
        ar["alone_busbw_gbs"] = round(2.0 * (world - 1) / world * ar["bytes"] / (ar["alone_ms"] * 1e-3) / 1e9, 1)
        # exposed: time from the end of backward to all buckets reduced
        grd, sat, gt, gwo, gor = resident
        exp = []
        for _ in range(4):
            reducer.zero_grad()
            out = model(grd, sat)
            l_ = losses.training_loss(out, gt, gwo, gor)
            l_.backward()
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b0.record()
            reducer.finish()
            b1.record()
            torch.cuda.synchronize()
            exp.append(b0.elapsed_time(b1))
            opt.step()
        ar["exposed_ms"] = round(min(exp), 3)
        ar["overlap"] = round(1.0 - ar["exposed_ms"] / ar["alone_ms"], 3) if ar["alone_ms"] > 0 else None
        step(resident)                              # gradients were left summed by the diagnostic: resync with a real step
    # ---- timed region: end to end from host buffers ----
    run_e2e(2)
    barrier()
    w0 = time.time()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run_e2e(args.steps)
    e1.record()
    barrier()
    sampler.window(w0, time.time())
    ms_e2e = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
    clocks = sampler.stop() if rank == 0 else None

    t = torch.tensor([ms_total, ms_e2e], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e = t.tolist()

    if rank == 0:
        peaks = B_._peaks()
        pt, ph = peaks["tensor_sustained"] * 1e12, peaks["hbm"] * 1e9
        pairs = world * Bsz * args.steps
        kern = {}
        for tag, r in layers.items():
            kname = tag.split(":")[0]
            k = kern.setdefault(kname, dict(launches=0, ms=0.0, flops=0.0, bytes=0.0, ideal_ms=0.0, tensor_ms=0.0))
            k["launches"] += r["launches"]
            k["ms"] += r["ms"]
            k["flops"] += r["flops"]
            k["bytes"] += r["bytes"]
            k["ideal_ms"] += max(r["flops"] / pt, r["bytes"] / ph) * 1e3
            if r["flops"] / pt > r["bytes"] / ph:
                k["tensor_ms"] += r["ms"]
        post_ms = sum(k["ms"] for k in kern.values())

        def describe(kname, k):
            sec = k["ms"] / 1e3
            tensor_bound = k["tensor_ms"] > 0.5 * k["ms"]
            if tensor_bound:
                ach, peak, unit = k["flops"] / sec / 1e12, peaks["tensor_sustained"], "TFLOP/s"
            else:
                ach, peak, unit = k["bytes"] / sec / 1e9, peaks["hbm"], "GB/s"
            return {"kernel": kname, "bound": "tensor" if tensor_bound else "hbm", "achieved": round(ach, 2), "peak": peak,
                    "unit": unit, "frac": round(ach / peak, 4), "frac_of_roofline_time": round(k["ideal_ms"] / k["ms"], 4),
                    "launches_per_step": k["launches"] // args.steps, "ms_per_step": round(k["ms"] / args.steps, 4),
                    "share_of_post_encoder_ms": round(k["ms"] / post_ms, 3), "traffic": None}

        kernels = {kname: describe(kname, k) for kname, k in sorted(kern.items(), key=lambda kv: -kv[1]["ms"])}
        dominant = max(kern.items(), key=lambda kv: kv[1]["ms"])[0]
        roofline = dict(kernels[dominant])
        roofline["peak_source"] = peaks["source"] + (" (sustained bf16)" if roofline["bound"] == "tensor" else " (copy)")
        roofline["post_encoder_ms_per_step"] = round(post_ms / args.steps, 3)
        roofline["note"] = ("achieved = algorithmic flops (2*M*N*K) or bytes of all launches of this kernel over the timed steps / "
                            "their CUDA-event time, from an eager pass with per-launch events right after the timed region")
        cpu = cpu_train_baseline(budget_s=40.0) if (world == 1 and not args.no_cpu) else None
        h2d = sum(t_.numel() * t_.element_size() for t_ in host)
        line = {
            "metric": METRIC, "value": round(pairs / (ms_total / 1e3), 3), "unit": "pairs/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms_total / args.steps, 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
            "config": {"workload": DESC, "workload_key": "train", "batch_per_gpu": Bsz, "global_batch": world * Bsz,
                       "parallelism": "data-parallel x%d (bucketed NCCL gradient all-reduce)" % world,
                       "backend": args.backend, "optimizer": "Adam(lr=1e-4, betas=(0.9, 0.999)), fused",
                       "encoder_memory_format": "channels_last", "cudnn_benchmark": True,
                       "cuda_graph": bool(use_graph), **({"cuda_graph_note": graph_note} if graph_note else {}),
                       "precision_note": "fp32 master weights and optimizer; encoders fp32 autograd; decoder activations and GEMM "
                                         "operands in the stated dtype with fp32 accumulation",
                       "l2": "per-step working set (>1 GB of saved activations) exceeds the 126 MB L2"},
            "post_encoder": {"ms_per_step": round(post_ms / args.steps, 3),
                             "note": "sum of the CUDA-event times of the libccvpe_b200 forward + backward kernels (rank 0)"},
            "e2e": {"value": round(pairs / (ms_e2e / 1e3), 3), "unit": "pairs/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": 4, "ms_per_step": round(ms_e2e / args.steps, 3),
                    "note": "images + ground-truth maps copied from pinned host memory every step (double buffered), the loss read "
                            "back on the host every step"},
            "gpu_launches": int(launches) * world, "final_loss": final_loss, "allreduce": ar,
            "roofline": roofline, "kernels": kernels, "clocks": clocks,
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
        if args.layers:
            with open(args.layers, "w") as f:
                f.write("%-72s %9s %10s %10s %9s\n" % ("kernel:family|layer", "ms/step", "TFLOP/s", "GB/s", "of-roof"))
                for tag, r in sorted(layers.items(), key=lambda kv: -kv[1]["ms"]):
                    sec = r["ms"] / 1e3
                    ideal = max(r["flops"] / pt, r["bytes"] / ph)
                    f.write("%-72s %9.4f %10.2f %10.1f %9.3f\n" % (tag, r["ms"] / args.steps, r["flops"] / sec / 1e12,
                                                                   r["bytes"] / sec / 1e9, ideal / sec))
    if dist is not None:
        # The captured training graph holds NCCL work: tearing the communicator down underneath it can block forever, so the
        # ranks meet at a barrier, flush and leave without running the process-group destructor.
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
