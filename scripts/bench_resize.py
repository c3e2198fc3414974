"""Device bilinear resize (models.resize_u8 / ccvpe_resize_u8): what it costs on the GPU and what it saves on the host.

  (a) kernel time (CUDA events) at B=64 for the VIGOR ground (1024x2048 -> 320x640) and aerial (640x640 -> 512x512)
      resizes from NHWC, and achieved GB/s of algorithmic bytes (read the input once, write the output once) against the
      6553.9 GB/s HBM peak of BASELINE.md.  `--iters` launches are captured in one CUDA graph and replayed under events.
      The ground batch (403 MB) exceeds the 126 MB L2; the aerial batch (79 MB) does not, so its later passes partly
      read from L2.
  (b) end to end, bf16 CVM_VIGOR B=64 in CUDA-graph mode, from pinned host uint8 images: per step H2D of both images, then
      forward + pose decode + D2H of the poses, software-pipelined like bench.py's e2e leg.  Once from native-resolution
      images with the resize on the device, once from images already at model resolution (bench.py's e2e input).  The
      un-overlapped H2D time of one step's native images is reported beside it.
  (c) Pillow's resize of one VIGOR pair on this host's CPU (one thread), the work the device resize takes off the host.

Prints one JSON object (with the GPU's name and power limit); `--out FILE` also writes it there."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

HBM_PEAK_GBS = 6553.9                   # BASELINE.md (MEASURED_PEAKS.json)
GROUND = ((1024, 2048), (320, 640))
AERIAL = ((640, 640), (512, 512))


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as exc:                                    # noqa: BLE001 -- reported, not fatal
        return {"name": torch.cuda.get_device_name(0), "nvidia_smi": "unavailable (%s)" % exc}


def kernel_time(B, src, dst, iters, dev):
    from ccvpe_b200 import models
    (H, W), (h, w) = src, dst
    x = torch.randint(0, 256, (B, H, W, 3), dtype=torch.uint8, device=dev)
    out = torch.empty((B, 3, h, w), dtype=torch.uint8, device=dev)
    for _ in range(3):
        models.CVM_VIGOR.resize_u8(x, dst, out=out)
    torch.cuda.synchronize()
    # the launches are captured in a CUDA graph, so the events time the kernels rather than the Python-side enqueue
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(iters):
            models.CVM_VIGOR.resize_u8(x, dst, out=out)
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    graph.replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    nbytes = x.numel() + out.numel()
    return {"B": B, "src": [H, W], "dst": [h, w], "layout": "NHWC", "us_per_call": round(ms * 1e3, 1),
            "algorithmic_bytes": nbytes, "gb_per_s": round(nbytes / ms / 1e6, 1),
            "share_of_hbm_peak": round(nbytes / ms / 1e6 / HBM_PEAK_GBS, 3)}


def end_to_end(B, steps, warmup, dev):
    from ccvpe_b200 import models
    from ccvpe_b200.synthetic import fill_deterministic

    model = models.CVM_VIGOR("cuda", True).eval()
    fill_deterministic(model.state_dict(), seed=0)
    model = model.to(dev).set_precision("bf16").set_cuda_graph(True)
    gen = torch.Generator().manual_seed(5)
    host = {"native": [torch.randint(0, 256, (B,) + s + (3,), generator=gen, dtype=torch.uint8).pin_memory()
                       for s in (GROUND[0], AERIAL[0])],
            "resized": [torch.randint(0, 256, (B, 3) + s, generator=gen, dtype=torch.uint8).pin_memory()
                        for s in (GROUND[1], AERIAL[1])]}
    dev_in = {k: [[torch.empty_like(t, device=dev) for t in v] for _ in range(2)] for k, v in host.items()}
    resized = [torch.empty((B, 3) + s, dtype=torch.uint8, device=dev) for s in (GROUND[1], AERIAL[1])]
    copy_stream = torch.cuda.Stream(device=dev)
    slot_free = [None, None]
    results = [None, None]

    def upload(kind, slot):
        with torch.cuda.stream(copy_stream):
            if slot_free[slot] is not None:
                copy_stream.wait_event(slot_free[slot])
            for d, h in zip(dev_in[kind][slot], host[kind]):
                d.copy_(h, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return ev

    def run(kind, n):
        """as bench.py's e2e leg: the copy of step i+1 is issued before step i computes, and the host reads the poses of
        step i-1 after it has enqueued step i"""
        slot_free[0] = slot_free[1] = None
        nxt, pending = upload(kind, 0), None
        for i in range(n):
            slot = i % 2
            ev = nxt
            if i + 1 < n:
                nxt = upload(kind, 1 - slot)
            torch.cuda.current_stream().wait_event(ev)
            g, s = dev_in[kind][slot]
            if kind == "native":
                g = model.resize_u8(g, GROUND[1], out=resized[0])
                s = model.resize_u8(s, AERIAL[1], out=resized[1])
            out = model(g, s)
            pose = model.decode_pose(out[1], out[2])
            slot_free[slot] = torch.cuda.Event()
            slot_free[slot].record()
            if results[slot] is None:
                results[slot] = {k: torch.empty(v.shape, dtype=v.dtype, pin_memory=True) for k, v in pose.items()}
            for k, v in pose.items():
                results[slot][k].copy_(v, non_blocking=True)
            done = torch.cuda.Event()
            done.record()
            if pending is not None:
                pending.synchronize()
            pending = done
        pending.synchronize()

    res = {}
    with torch.no_grad():
        for kind in ("native", "resized"):
            run(kind, warmup)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run(kind, steps)
            torch.cuda.synchronize()
            ms = (time.perf_counter() - t0) * 1e3 / steps
            res[kind] = {"ms_per_step": round(ms, 3), "pairs_per_s": round(B / ms * 1e3, 1),
                         "h2d_bytes_per_step": sum(t.numel() for t in host[kind])}
        for kind in ("native", "resized"):                   # one step's H2D alone, not overlapped with anything
            upload(kind, 0)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.cuda.current_stream().wait_event(upload(kind, 0))
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            res[kind].update(h2d_alone_ms=round(ms, 3), h2d_gb_per_s=round(res[kind]["h2d_bytes_per_step"] / ms / 1e6, 1))
    res.update(B=B, model="CVM_VIGOR bf16, CUDA graph", steps=steps)
    return res


def host_pillow(pairs):
    from PIL import Image
    rng = np.random.default_rng(0)
    g = [Image.fromarray(rng.integers(0, 256, GROUND[0] + (3,), dtype=np.uint8)) for _ in range(pairs)]
    s = [Image.fromarray(rng.integers(0, 256, AERIAL[0] + (3,), dtype=np.uint8)) for _ in range(pairs)]
    g[0].resize(GROUND[1][::-1], Image.BILINEAR)
    t = {}
    for name, imgs, size in (("ground", g, GROUND[1]), ("aerial", s, AERIAL[1])):
        t0 = time.perf_counter()
        for im in imgs:
            im.resize(size[::-1], Image.BILINEAR)
        t[name] = (time.perf_counter() - t0) * 1e3 / pairs
    import PIL
    return {"pillow": PIL.__version__, "threads": 1, "cpu_count": os.cpu_count(),
            "ground_ms": round(t["ground"], 2), "aerial_ms": round(t["aerial"], 2),
            "ms_per_pair": round(t["ground"] + t["aerial"], 2)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--iters", type=int, default=50, help="kernel-time launches per shape")
    ap.add_argument("--steps", type=int, default=20, help="timed end-to-end steps per input kind")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--pairs", type=int, default=10, help="pairs resized with Pillow on the host")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_resize.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    res = {"gpu": gpu_info(),
           "kernel": {"ground": kernel_time(args.batch, *GROUND, args.iters, dev),
                      "aerial": kernel_time(args.batch, *AERIAL, args.iters, dev)},
           "e2e": end_to_end(args.batch, args.steps, args.warmup, dev),
           "host": host_pillow(args.pairs)}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
