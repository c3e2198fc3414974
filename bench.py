#!/usr/bin/env python
"""bench.py -- VIGOR pairs/sec of the CCVPE hot path on N B200s (BASELINE.json metric), one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload W] [--batch B] [--scaling weak|strong]
                    [--precision bf16|fp32] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of `CVM_VIGOR.forward` + pose decode over one batch of synthetic VIGOR-shaped pairs
(3x320x640 panorama + 3x512x512 aerial, random-init weights).  Workload = BASELINE.json configs[1]: batch 64 bf16 per
GPU, batch-sharded (weak scaling: every rank owns its own 64 pairs; no data-path collective -- pairs are independent).

  value     : pairs/s, inputs resident in HBM, K steps timed with CUDA events between barrier+synchronize, max over ranks
  e2e       : same metric through the public API with HOST (pinned) inputs: H2D copy of both images and D2H read of the
              decoded poses inside the timed region, every step
  roofline  : the dominant kernel family of the post-encoder path, timed live with CUDA events on the launch stream
  kernels   : per-family achieved GB/s or TFLOP/s vs the measured peaks (MEASURED_PEAKS.json)
  cpu_baseline : the oracle port of the reference's CPU forward, timed on the host cores on a bounded sample (rank 0)

  parity    : the timed bf16 outputs of the first 8 pairs against this library's exact-fp32 path (argmax agreement, errors)
  torch_gpu_baseline : the reference's op sequence through PyTorch's own GPU kernels on the same B200 (fp32 / bf16 autocast)

Other workloads (`--workload kitti_b32 | vigor_prior72_fov180 | vigor_prior72_fov108 | oxford_b1 | train`) print the same
line for BASELINE.json configs 3-5 and the Oxford batch-1 latency; `--scaling strong` shards ONE global batch.

`--impl reference` times the reference's CPU forward (the unmodified reference when a copy sits in baseline/_ref/, else the
oracle port that the tests pin bit-equal to it) and prints the same line with "impl": "reference".
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "VIGOR pairs/sec (CVM_VIGOR forward + pose decode, 320x640 panorama + 512x512 aerial)"

#: --workload: the BASELINE.json configurations.  `vigor_b64` (configs[1]) is the one the metric is quoted on and the
#: default; the others are configs[2] (KITTI), configs[3] (limited FoV + orientation prior) and the reference's one published
#: speed figure (Oxford RobotCar, batch-1 sequential frames, README.md:19); `train` is configs[4] (bench_train.py).
WORKLOADS = {
    "vigor_b64": dict(cls="CVM_VIGOR", variant="vigor", ground=(320, 640), circular=True, ori_noise=None, batch=64,
                      metric=METRIC,
                      desc="CVM_VIGOR batched inference, synthetic VIGOR shape (3x320x640 + 3x512x512), FoV 360, "
                           "random-init weights (BASELINE.json configs[1])"),
    "kitti_b32": dict(cls="CVM_KITTI", variant="kitti", ground=(256, 1024), circular=None, ori_noise=None, batch=32,
                      metric="KITTI pairs/sec (CVM_KITTI forward + pose decode, 256x1024 ground + 512x512 aerial)",
                      desc="CVM_KITTI batched inference, synthetic KITTI shape (3x256x1024 + 3x512x512), 16 orientations, "
                           "random-init weights (BASELINE.json configs[2])"),
    "vigor_prior72_fov180": dict(cls="CVM_VIGOR_ori_prior", variant="vigor_prior", ground=(320, 320), circular=False,
                                 ori_noise=72.0, batch=64,
                                 metric="VIGOR limited-FoV pairs/sec (CVM_VIGOR_ori_prior(72) forward + pose decode, FoV 180: "
                                        "320x320 panorama crop + 512x512 aerial)",
                                 desc="CVM_VIGOR_ori_prior(ori_noise=72) batched inference, FoV 180 (panorama cropped to 320x320), "
                                      "9 orientations per level (BASELINE.json configs[3])"),
    "vigor_prior72_fov108": dict(cls="CVM_VIGOR_ori_prior", variant="vigor_prior", ground=(320, 192), circular=False,
                                 ori_noise=72.0, batch=64,
                                 metric="VIGOR limited-FoV pairs/sec (CVM_VIGOR_ori_prior(72) forward + pose decode, FoV 108: "
                                        "320x192 panorama crop + 512x512 aerial)",
                                 desc="CVM_VIGOR_ori_prior(ori_noise=72) batched inference, FoV 108 (panorama cropped to 320x192), "
                                      "9 orientations per level (BASELINE.json configs[3])"),
    "oxford_b1": dict(cls="CVM_OxfordRobotCar", variant="oxford", ground=(154, 231), circular=None, ori_noise=None, batch=1,
                      metric="Oxford RobotCar frames/sec (CVM_OxfordRobotCar forward + pose decode, batch 1, sequential frames)",
                      desc="CVM_OxfordRobotCar sequential per-frame inference, batch 1 (3x154x231 + 3x512x512); the reference "
                           "publishes 14 FPS on an unstated GPU (README.md:19, loop train_OxfordRobotCar.py:195-246)"),
}


def build_workload_model(wl, device="cpu"):
    from ccvpe_b200 import models
    cls = getattr(models, wl["cls"])
    if wl["cls"] == "CVM_VIGOR":
        return cls(device, wl["circular"])
    if wl["cls"] == "CVM_VIGOR_ori_prior":
        return cls(device, wl["ori_noise"], wl["circular"])
    return cls(device)


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], tensor_burst=p["bf16_tflops"], tensor_sustained=p["bf16_tflops_sustained"],
                    source="measured")
    return dict(hbm=6650.0, tensor_burst=1590.0, tensor_sustained=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms (B200_PROFILING.md); only samples whose timestamp falls
    inside a timed window are used."""
    QUERY = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []
        self.windows = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)             # the sampler never outlives a run that stops early
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def window(self, t0: float, t1: float):
        self.windows.append((t0, t1))

    def stop(self):
        import datetime

        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                clk, cmax = float(f[1]), float(f[2])
            except ValueError:
                continue
            if not any(t0 - 0.05 <= ts <= t1 + 0.05 for t0, t1 in self.windows):
                continue
            sm.append(clk)
            smax.append(cmax)
            try:
                power.append(float(f[3]))
            except ValueError:
                pass
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples inside the timed windows"],
                    "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


# ---------------------------------------------------------------------------------------------------------------------
# CPU baseline: oracle port of the reference forward (encoders are PyTorch in both)
# ---------------------------------------------------------------------------------------------------------------------
def _real_reference_module():
    """The UNMODIFIED reference, if a copy travelled to this box under baseline/_ref/ (git-ignored; the driver or a
    maintainer may place it there -- this repo never copies it).  Returns the reference's `models` module or None."""
    root = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isfile(os.path.join(root, "models.py")):
        return None
    try:
        from oracle import ref_shim
        ref_shim.REFERENCE_ROOT = root
        return ref_shim.load_reference_models()
    except Exception as exc:                                    # noqa: BLE001 -- fall back to the pinned port
        print("bench.py: baseline/_ref present but not importable (%s); timing the oracle port" % exc, file=sys.stderr)
        return None


def cpu_reference_throughput(wl, sample_batch: int, reps: int, budget_s: float = 30.0):
    """The reference's CPU forward + numpy pose decode on the host cores: the real reference when baseline/_ref holds it
    (kind "reference"), else the oracle port, which tests pin bit-equal to the reference (kind "port")."""
    from ccvpe_b200.synthetic import fill_deterministic, synthetic_pair
    from oracle import ccvpe_oracle as orc

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    model = build_workload_model(wl, "cpu").eval()
    fill_deterministic(model.state_dict(), seed=0)
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    grd, sat = synthetic_pair(sample_batch, wl["ground"], seed=0)
    ref_mod = _real_reference_module()
    ref_model = None
    if ref_mod is not None:
        cls = getattr(ref_mod, wl["cls"])
        if wl["cls"] == "CVM_VIGOR":
            ref_model = cls("cpu", wl["circular"])
        elif wl["cls"] == "CVM_VIGOR_ori_prior":
            ref_model = cls("cpu", wl["ori_noise"], wl["circular"])
        else:
            ref_model = cls("cpu")
        ref_model.load_state_dict(sd, strict=True)
        ref_model.eval()
    times = []
    t_begin = time.time()
    with torch.no_grad():
        for i in range(reps + 1):
            t0 = time.time()
            if ref_model is not None:
                out = ref_model(grd, sat)
            else:
                out = orc.forward_full(wl["variant"], sd, model.grd_efficientnet, model.sat_efficientnet, grd, sat,
                                       wl["ori_noise"])
            orc.pose_decode(out[1].numpy(), out[2].numpy())
            dt = time.time() - t0
            if i > 0:
                times.append(dt)            # first pass is the warm-up
            if time.time() - t_begin > budget_s and times:
                break
    best = min(times)
    what = "unmodified reference (baseline/_ref)" if ref_model is not None else "oracle port"
    return dict(value=sample_batch / best, unit="pairs/s", cores=cores, kind="reference" if ref_model is not None else "port",
                sample="%s of %s.forward + numpy pose decode, fp32, batch %d, best of %d after 1 warm-up "
                       "(%.2f s/forward, torch threads=%d)" % (what, wl["cls"], sample_batch, len(times), best, cores))


def torch_gpu_baseline(wl, dev, sample_batch: int):
    """BASELINE.md section 3: the reference's own arithmetic through PyTorch's library kernels (cuDNN / cuBLAS / ATen) on
    this same B200 -- the oracle port's torch ops executed on the GPU, fp32 with TF32 off and under bf16 autocast.  A
    reported comparator (what `model.cuda()` of the reference would give), never part of the product path."""
    from ccvpe_b200.synthetic import fill_deterministic, synthetic_pair
    from oracle import ccvpe_oracle as orc

    model = build_workload_model(wl, "cuda").eval()
    fill_deterministic(model.state_dict(), seed=0)
    model = model.to(dev)
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    grd, sat = (t.to(dev) for t in synthetic_pair(sample_batch, wl["ground"], seed=0))
    out = {}

    def once():
        o = orc.forward_full(wl["variant"], sd, model.grd_efficientnet, model.sat_efficientnet, grd, sat, wl["ori_noise"])
        return o[1].flatten(1).argmax(dim=1)

    for tag, ctx in (("fp32_tf32_off", torch.backends.cudnn.flags(enabled=True, allow_tf32=False)),
                     ("bf16_autocast", torch.autocast("cuda", dtype=torch.bfloat16))):
        try:
            with torch.no_grad(), ctx:
                once()
                torch.cuda.synchronize()
                best = None
                for _ in range(3):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    once()
                    e1.record()
                    torch.cuda.synchronize()
                    ms = e0.elapsed_time(e1)
                    best = ms if best is None else min(best, ms)
            out[tag] = {"value": round(sample_batch / (best / 1e3), 2), "unit": "pairs/s", "ms_per_forward": round(best, 3)}
        except Exception as exc:                                # noqa: BLE001
            out[tag] = {"error": "%s: %s" % (type(exc).__name__, exc)}
    out["sample"] = ("oracle port of %s.forward (the reference's op sequence) through cuDNN/cuBLAS/ATen on this GPU, batch %d, "
                     "inputs resident, best of 3 after 1 warm-up; argmax on the device" % (wl["cls"], sample_batch))
    del model, sd
    torch.cuda.empty_cache()
    return out


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    reps = max(1, min(args.steps, 10))
    base = cpu_reference_throughput(wl, sample_batch=1, reps=reps + args.warmup, budget_s=120.0)
    line = {
        "impl": "reference", "metric": wl["metric"], "value": base["value"], "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 / base["value"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["desc"] + " -- CPU arm: bounded sample of batch 1 per step", "workload_key": args.workload,
                   "batch_per_gpu": args.batch or wl["batch"], "parallelism": "cpu"},
        "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------------------
OUT_NAMES = ["logits", "heatmap", "ori", "scores1", "scores2", "scores3", "scores4", "scores5", "scores6"]
#: --dump-outputs stores an array of up to this many elements whole and a sample of this many elements of a larger one, so
#: one step's 9 outputs and 5 pose fields stay well under 64 MB
DUMP_MAX_ELEMS = 1 << 20


def host_outputs(out, pose):
    """What one step hands its caller -- the 9 forward outputs and the decoded poses (`pose_<field>`) -- as host float32
    (floating-point tensors) or float64 (integer tensors, exact) arrays.  A larger array becomes the elements at a fixed,
    seeded set of sorted flat indices, the same set in every run with the same arguments."""
    import numpy as np

    arrays = dict(zip(OUT_NAMES, out), **{"pose_" + k: v for k, v in pose.items()})
    host = {}
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_MAX_ELEMS:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_MAX_ELEMS, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        dtype = torch.float32 if t.is_floating_point() and t.dtype != torch.float64 else torch.float64
        host[name] = t.to(dtype).cpu().numpy()
    return host


def run_ours(args):
    from ccvpe_b200 import cabi, models
    from ccvpe_b200.decoder import OpTimer
    from ccvpe_b200.synthetic import fill_deterministic, synthetic_pair

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        # keep stdout to the one JSON line: NCCL prints its version banner to stdout when the first communicator is
        # created (at NCCL_DEBUG=VERSION/WARN/INFO, whatever the box sets), so route fd 1 to stderr around the
        # rendezvous and the first collective
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

    wl = WORKLOADS[args.workload]
    global_batch = args.batch or wl["batch"]
    if args.scaling == "strong":
        # BASELINE.json configs[1] read literally: ONE batch of `global_batch` pairs sharded over the ranks
        from ccvpe_b200.sharding import shard_bounds
        lo, hi = shard_bounds(global_batch, rank, world)
        B = hi - lo
        if B == 0:
            raise SystemExit("strong scaling: global batch %d < world size %d" % (global_batch, world))
    else:
        B = global_batch
    model = build_workload_model(wl, "cuda").eval()
    fill_deterministic(model.state_dict(), seed=0)
    model = model.to(dev).set_precision(args.precision)
    if args.backend == "simt":
        model.set_backend(cabi.BACKEND_SIMT)
    grd_h, sat_h = synthetic_pair(B, wl["ground"], seed=100 + rank)
    grd_h, sat_h = grd_h.pin_memory(), sat_h.pin_memory()
    grd_d, sat_d = grd_h.to(dev), sat_h.to(dev)
    # uint8 host images for the end-to-end leg (what an image decoder hands over): ingest = ToTensor + ImageNet Normalize on
    # the device (models.ingest, reference train_VIGOR.py:55-70); 4x fewer H2D bytes than the reference's fp32 tensors
    gen8 = torch.Generator().manual_seed(300 + rank)
    grd_u8 = torch.randint(0, 256, tuple(grd_h.shape), generator=gen8, dtype=torch.uint8).pin_memory()
    sat_u8 = torch.randint(0, 256, tuple(sat_h.shape), generator=gen8, dtype=torch.uint8).pin_memory()

    def step_resident():
        out = model(grd_d, sat_d)
        return out, model.decode_pose(out[1], out[2])

    copy_stream = torch.cuda.Stream(device=dev)
    # e2e: two preallocated device input slots (no allocator traffic inside the timed region): the H2D copy of step i+1
    # lands in the slot step i-1 used, guarded by an event recorded when that step's kernels were enqueued
    host_in = {"fp32": (grd_h, sat_h), "uint8": (grd_u8, sat_u8)}
    dev_in = {k: [(torch.empty(v[0].shape, dtype=v[0].dtype, device=dev), torch.empty(v[1].shape, dtype=v[1].dtype, device=dev))
                  for _ in range(2)] for k, v in host_in.items()}
    ingest_out = (torch.empty_like(grd_d), torch.empty_like(sat_d))
    slot_free = [None, None]
    e2e_input = ["uint8"]

    def upload(slot):
        """H2D of one step's inputs from pinned host memory on the copy stream; returns the copy-done event."""
        kind = e2e_input[0]
        with torch.cuda.stream(copy_stream):
            if slot_free[slot] is not None:
                copy_stream.wait_event(slot_free[slot])
            dev_in[kind][slot][0].copy_(host_in[kind][0], non_blocking=True)
            dev_in[kind][slot][1].copy_(host_in[kind][1], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return ev

    def e2e_forward(slot):
        g_in, s_in = dev_in[e2e_input[0]][slot]
        if e2e_input[0] == "uint8" and args.precision != "bf16":
            g_in = model.ingest(g_in, out=ingest_out[0])
            s_in = model.ingest(s_in, out=ingest_out[1])
        return model(g_in, s_in)         # (bf16 plan: uint8 is normalised inside the stem kernel's loads)

    host_results = [None, None]      # double-buffered pinned host copies of the pose tensors

    def run_e2e(steps):
        """Every step: H2D copy of its inputs + forward + pose decode + D2H read of the poses.  Software-pipelined like a
        serving loop: the copy of step i+1 is issued before step i computes (double buffering) and the host reads the
        poses of step i-1 after it has enqueued step i, so the GPU never drains between steps; nothing is reused across
        steps and every step's result is read on the host inside the timed region."""
        nxt = upload(0)
        pending = None
        last = None
        for i in range(steps):
            slot = i % 2
            ev = nxt
            if i + 1 < steps:
                nxt = upload(1 - slot)
            torch.cuda.current_stream().wait_event(ev)
            out = e2e_forward(slot)
            pose = model.decode_pose(out[1], out[2])
            slot_free[slot] = torch.cuda.Event()
            slot_free[slot].record()
            if host_results[slot] is None:
                host_results[slot] = {k: torch.empty(v.shape, dtype=v.dtype, pin_memory=True) for k, v in pose.items()}
            for k, v in pose.items():
                host_results[slot][k].copy_(v, non_blocking=True)           # D2H of the step's result
            done = torch.cuda.Event()
            done.record()
            if pending is not None:                                           # host-side read of the previous step's poses
                pending[1].synchronize()
                last = {k: v.clone() for k, v in pending[0].items()}
            pending = (host_results[slot], done)
        pending[1].synchronize()
        last = {k: v.clone() for k, v in pending[0].items()}
        return last

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ncu_range = bool(os.environ.get("CCVPE_NCU_RANGE"))         # `ncu --profile-from-start off`: capture exactly these steps
    use_graph = not (args.no_cuda_graph or ncu_range)
    graph_note = None
    with torch.no_grad():
        for _ in range(2):
            step_resident()                                     # eager: builds weight caches and staging buffers
        if use_graph:
            # the model's CUDA-graph mode (models.set_cuda_graph): the ~200 launches of a forward replay as one graph
            try:
                model.set_cuda_graph(True)
                step_resident()
                torch.cuda.synchronize()
            except Exception as exc:                            # capture is an optimisation, never a requirement
                model.set_cuda_graph(False)
                use_graph = False
                graph_note = "CUDA-graph capture failed (%s: %s); ran eagerly" % (type(exc).__name__, exc)
        for _ in range(max(args.warmup, 3)):
            step_resident()
        barrier()
        # ---- timed region: device-resident inputs ------------------------------------------------------------
        timer = OpTimer()
        if not use_graph:
            model.pipeline.timer = timer                        # eager: per-launch events inside the timed region
        cabi.reset_launch_count()
        barrier()
        w0 = time.time()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if ncu_range:
            torch.cuda.profiler.start()
        ev0.record()
        for _ in range(args.steps):
            last = step_resident()
        ev1.record()
        if ncu_range:
            torch.cuda.synchronize()
            torch.cuda.profiler.stop()
        barrier()
        sampler.window(w0, time.time())
        # copied now: in CUDA-graph mode the outputs are the graph's static buffers, which every later forward overwrites
        dumped = host_outputs(*last) if args.dump_outputs and rank == 0 else None
        launches = cabi.launch_count()
        ms_total = ev0.elapsed_time(ev1)
        if use_graph:
            # a replayed graph leaves no per-kernel events: attribute time to kernels with an eager pass over the same
            # steps right after the timed region (same kernels, same inputs; with a timer set, forward runs eagerly)
            model.pipeline.timer = timer
            for _ in range(args.steps):
                step_resident()
            torch.cuda.synchronize()
        layers = timer.summary()
        model.pipeline.timer = None
        # ---- timed region: end to end from host buffers ------------------------------------------------------
        h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e2e_input[0] = args.e2e_input
        upload(0)                                       # first use of the copy stream: not representative
        torch.cuda.synchronize()
        h0.record()
        _ev = upload(0)
        torch.cuda.current_stream().wait_event(_ev)
        h1.record()
        torch.cuda.synchronize()
        h2d_ms = h0.elapsed_time(h1)                    # diagnostic: one un-overlapped H2D copy of a step's inputs
        def timed_e2e(kind):
            e2e_input[0] = kind
            slot_free[0] = slot_free[1] = None
            run_e2e(2)
            barrier()
            w0_ = time.time()
            t0 = time.perf_counter()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run_e2e(args.steps)
            e1.record()
            barrier()
            sampler.window(w0_, time.time())
            return max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)

        ms_e2e_f32 = timed_e2e("fp32")               # the reference's own hand-over: fp32 tensors from the DataLoader
        ms_e2e = timed_e2e(args.e2e_input)           # headline: uint8 images + device-side ingest (default)
        clocks = sampler.stop() if rank == 0 else None
        # ---- parity of the timed path (rank 0): the bf16 tcgen05 outputs of the first pairs of the timed batch against
        # the fp32 parity path (exact-fp32 CUDA-core kernels + fp32 encoders, itself <= 1e-3 from the oracle: tests/)
        parity = None
        if rank == 0 and args.precision == "bf16" and not args.no_parity:
            n_par = min(8, B)
            model.set_cuda_graph(False)
            o16 = [t.clone() for t in model(grd_d[:n_par], sat_d[:n_par])]
            model.set_precision("fp32")
            o32 = model(grd_d[:n_par], sat_d[:n_par])
            torch.cuda.synchronize()
            model.set_precision(args.precision)

            def _rel(a, b):
                return float((a - b).abs().max() / b.abs().max())

            def _rms(a, b):
                return float((a - b).double().pow(2).mean().sqrt() / b.double().pow(2).mean().sqrt())

            am16, am32 = o16[1].flatten(1).argmax(dim=1), o32[1].flatten(1).argmax(dim=1)
            top = torch.topk(o32[0], 2, dim=1).values
            logit_rms = float((o16[0] - o32[0]).pow(2).mean().sqrt())
            decided = (top[:, 0] - top[:, 1]) > 10 * logit_rms
            cosang = (o16[2] * o32[2]).sum(dim=1).clamp(-1, 1)
            parity = {"pairs": n_par, "against": "fp32 parity path of this library on the same pairs (SIMT kernels, fp32 encoders)",
                      "argmax_agree": int((am16 == am32).sum()), "argmax_decided_pairs": int(decided.sum()),
                      "argmax_agree_decided": int(((am16 == am32) & decided).sum()),
                      "logits_max_rel_err": round(_rel(o16[0], o32[0]), 5), "logits_rms_rel_err": round(_rms(o16[0], o32[0]), 5),
                      "heatmap_max_rel_err": round(_rel(o16[1], o32[1]), 5),
                      "scores_max_rel_err": [round(_rel(a, b), 5) for a, b in zip(o16[3:], o32[3:])],
                      "ori_angle_deg_median": round(float(torch.rad2deg(torch.acos(cosang)).median()), 4),
                      "stated_bf16_tolerance": "vs the fp32 CPU oracle at the benchmarked sizes (tests/test_gpu_forward.py, measured in "
                                               "profiles/r02_parity.md): max 4e-2 of max|ref|, rms 3e-2 of rms(ref) per tensor"}
            del o16, o32

    t = torch.tensor([ms_total, ms_e2e, ms_e2e_f32], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e, ms_e2e_f32 = t.tolist()

    if rank == 0:
        peaks = _peaks()
        pt, ph = peaks["tensor_sustained"] * 1e12, peaks["hbm"] * 1e9
        pairs_per_step = global_batch if args.scaling == "strong" else world * B
        pairs = pairs_per_step * args.steps
        value = pairs / (ms_total / 1e3)
        e2e_value = pairs / (ms_e2e / 1e3)
        # tags are "kernel:family|layer"; every layer has one shape, so its bound follows from its arithmetic intensity
        kern = {}
        for tag, r in layers.items():
            kname = tag.split(":")[0]
            k = kern.setdefault(kname, dict(launches=0, ms=0.0, flops=0.0, bytes=0.0, ideal_ms=0.0, tensor_ms=0.0))
            ideal = max(r["flops"] / pt, r["bytes"] / ph) * 1e3
            k["launches"] += r["launches"]
            k["ms"] += r["ms"]
            k["flops"] += r["flops"]
            k["bytes"] += r["bytes"]
            k["ideal_ms"] += ideal
            if r["flops"] / pt > r["bytes"] / ph:
                k["tensor_ms"] += r["ms"]
        post_ms = sum(k["ms"] for k in kern.values())
        traffic = {}
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            traffic = json.load(open(tpath))

        def describe(kname, k):
            sec = k["ms"] / 1e3
            tensor_bound = k["tensor_ms"] > 0.5 * k["ms"]
            if tensor_bound:
                ach, peak, unit = k["flops"] / sec / 1e12, peaks["tensor_sustained"], "TFLOP/s"
            else:
                ach, peak, unit = k["bytes"] / sec / 1e9, peaks["hbm"], "GB/s"
            return {"kernel": kname, "bound": "tensor" if tensor_bound else "hbm", "achieved": round(ach, 2),
                    "peak": peak, "unit": unit, "frac": round(ach / peak, 4),
                    "frac_of_roofline_time": round(k["ideal_ms"] / k["ms"], 4),
                    "launches_per_step": k["launches"] // args.steps, "ms_per_step": round(k["ms"] / args.steps, 4),
                    "share_of_post_encoder_ms": round(k["ms"] / post_ms, 3),
                    "traffic": traffic.get(kname)}

        kernels = {kname: describe(kname, k) for kname, k in sorted(kern.items(), key=lambda kv: -kv[1]["ms"])}
        dominant = max(kern.items(), key=lambda kv: kv[1]["ms"])[0]
        roofline = dict(kernels[dominant])
        roofline["peak_source"] = peaks["source"] + (" (sustained bf16)" if roofline["bound"] == "tensor" else " (copy)")
        roofline["post_encoder_ms_per_step"] = round(post_ms / args.steps, 3)
        roofline["note"] = ("achieved = algorithmic bytes (inputs + weights + outputs, each once) or 2*M*N*K flops of all "
                            "launches of this kernel over the timed steps / their CUDA-event time"
                            + ("; the timed region replays each forward as ONE CUDA graph (no per-kernel events), so the "
                               "per-launch events come from an eager pass over the same steps right after it"
                               if use_graph else ""))
        cpu = cpu_reference_throughput(wl, sample_batch=1, reps=5, budget_s=25.0) if (world == 1 and not args.no_cpu) else None
        gpu_base = None
        if world == 1 and not args.no_cpu and not args.no_torch_gpu_baseline:
            try:
                gpu_base = torch_gpu_baseline(wl, dev, sample_batch=min(B, 16))
            except Exception as exc:                            # noqa: BLE001 -- a comparator must never sink the bench line
                gpu_base = {"error": "%s: %s" % (type(exc).__name__, exc)}
        h2d_f32 = grd_h.numel() * grd_h.element_size() + sat_h.numel() * sat_h.element_size()
        h2d = h2d_f32 if args.e2e_input == "fp32" else grd_u8.numel() + sat_u8.numel()
        d2h = B * (8 + 8 + 8 + 8 + 1)
        line = {
            "metric": wl["metric"], "value": round(value, 3), "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": round(ms_total / args.steps, 3), "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "f32",
            "data": "synthetic",
            "config": {"workload": wl["desc"], "workload_key": args.workload,
                       "batch_per_gpu": B, "global_batch": pairs_per_step, "parallelism": "batch-sharded x%d" % world,
                       "backend": args.backend,
                       "cuda_graph": bool(use_graph), **({"cuda_graph_note": graph_note} if graph_note else {}),
                       "l2": "per-step working set (inputs %.0f MB + >1 GB activations) exceeds the 126 MB L2" % (h2d_f32 / 1e6)},
            # SURVEY section 8(d): the post-encoder path on its own (sum of the per-launch CUDA-event times of the
            # libccvpe_b200 decoder kernels, encoders excluded)
            "post_encoder": {"value": round(B * args.steps / (post_ms / 1e3), 1), "unit": "pairs/s per GPU (rank 0)",
                             "ms_per_step": round(post_ms / args.steps, 3)},
            "e2e": {"value": round(e2e_value, 3), "unit": "pairs/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": round(ms_e2e / args.steps, 3),
                    "h2d_alone_ms": round(h2d_ms, 3), "h2d_gbs": round(h2d / h2d_ms / 1e6, 1), "input": args.e2e_input,
                    "note": ("uint8 host images (what an image decoder produces) from pinned memory, ToTensor + ImageNet Normalize "
                             "on the device, fused into the stem kernel's loads" if args.e2e_input == "uint8" else
                             "fp32 host images from pinned memory") +
                            "; the H2D copy of step i+1 overlaps the kernels of step i and the host reads step i-1's poses "
                            "(pinned D2H) after enqueuing step i",
                    "fp32_host_images": {"value": round(pairs / (ms_e2e_f32 / 1e3), 3), "ms_per_step": round(ms_e2e_f32 / args.steps, 3),
                                         "h2d_bytes_per_step": h2d_f32,
                                         "note": "same loop with the reference's own hand-over (fp32 tensors, train_VIGOR.py:268-270)"}},
            "gpu_launches": int(launches) * world,      # libccvpe_b200 kernel launches in the timed region, all ranks
            "roofline": roofline, "kernels": kernels, "clocks": clocks,
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if gpu_base is not None:
            line["torch_gpu_baseline"] = gpu_base
        if parity is not None:
            line["parity"] = parity
        if B == 1:
            line["latency_ms_per_frame"] = {"resident": round(ms_total / args.steps, 3), "e2e": round(ms_e2e / args.steps, 3),
                                            "reference_published_fps": 14.0 if args.workload == "oxford_b1" else None}
        print(json.dumps(line), flush=True)
        if args.layers:
            with open(args.layers, "w") as f:
                f.write("%-64s %9s %10s %10s %9s\n" % ("kernel:family|layer", "ms/step", "TFLOP/s", "GB/s", "of-roof"))
                for tag, r in sorted(layers.items(), key=lambda kv: -kv[1]["ms"]):
                    sec = r["ms"] / 1e3
                    ideal = max(r["flops"] / pt, r["bytes"] / ph)
                    f.write("%-64s %9.4f %10.2f %10.1f %9.3f\n" % (tag, r["ms"] / args.steps, r["flops"] / sec / 1e12,
                                                                   r["bytes"] / sec / 1e9, ideal / sec))
        if dumped is not None:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dumped.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="vigor_b64", choices=sorted(WORKLOADS) + ["train"])
    ap.add_argument("--batch", type=int, default=0, help="pairs per GPU per step (weak) / global batch (strong); "
                                                         "default: the workload's (64 VIGOR, 32 KITTI, 1 Oxford)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: every rank owns its own batch; strong: ONE global batch sharded over the ranks")
    ap.add_argument("--e2e-input", default="uint8", choices=["uint8", "fp32"],
                    help="host image format of the end-to-end leg (the fp32 variant is always reported next to it)")
    ap.add_argument("--no-parity", action="store_true", help="skip the bf16-vs-fp32 parity record")
    ap.add_argument("--no-torch-gpu-baseline", action="store_true", help="skip the PyTorch-on-GPU comparator leg")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--backend", default="auto", choices=["auto", "simt"])
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-cuda-graph", action="store_true", help="launch every kernel eagerly in the timed regions")
    ap.add_argument("--layers", default=None, help="write a per-layer timing table to this file")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last timed step computed (rank 0) as DIR/<name>.npy, to compare two builds output "
                         "for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload == "train" or args.impl == "reference"):
        ap.error("--dump-outputs covers the inference workloads of --impl ours")
    if args.workload == "train":
        import bench_train
        bench_train.main(args)
    elif args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
