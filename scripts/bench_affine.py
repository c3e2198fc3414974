"""Device bilinear affine transform (models.affine_u8 / rotate_u8, ccvpe_affine_u8): what it costs on the GPU and what it
saves on the host.

  (a) kernel time (CUDA events around one replay of a CUDA graph of `--iters` launches) at B=64, NHWC input, a different
      rotation per image, for
        rot512:   512x512 -> 512x512 rotation about the centre (an aerial orientation augmentation);
        crop1280: 1280x1280 -> 512x512 rotation about the centre + centre crop (rotate a larger tile, keep the middle).
      Achieved GB/s of algorithmic bytes: every source pixel some output pixel's bilinear taps read (counted on the host
      from the same arithmetic), read once, plus the output written once; and that rate's share of the 6553.9 GB/s HBM
      peak of BASELINE.md.  The launches cycle through 3 input and 3 output buffers (> 126 MB L2 per cycle for both
      shapes), so the L2 does not carry an input from one launch to the next.
  (b) Pillow's cost per image on this host's CPU (one thread) for the same operations: Image.rotate(angle, BILINEAR) of a
      512x512 image, and for the 1280x1280 tile both Image.rotate(..).crop(box) and the cheapest exact host form,
      Image.transform((896, 896), AFFINE, m, BILINEAR).crop(box).

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
#: name -> (source (H, W), output (h, w), crop offset (left, top))
SHAPES = {"rot512": ((512, 512), (512, 512), (0, 0)), "crop1280": ((1280, 1280), (512, 512), (384, 384))}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as exc:                                    # noqa: BLE001 -- reported, not fatal
        return {"name": torch.cuda.get_device_name(0), "nvidia_smi": "unavailable (%s)" % exc}


def angles(B):
    return [float(a) for a in np.random.default_rng(7).uniform(-180.0, 180.0, B)]


def footprint_pixels(m, src, size, offset):
    """Distinct source pixels read by the bilinear taps of one image's inside output pixels (the kernel's arithmetic in
    numpy float64; the taps' clamping included)."""
    (H, W), (h, w), (left, top) = src, size, offset
    x = np.arange(left, left + w, dtype=np.float64)[None, :] + 0.5
    y = np.arange(top, top + h, dtype=np.float64)[:, None] + 0.5
    xi, yi = m[0] * x + m[1] * y + m[2], m[3] * x + m[4] * y + m[5]
    inside = (xi >= 0) & (xi < W) & (yi >= 0) & (yi < H)
    xf, yf = np.floor(xi[inside] - 0.5).astype(np.int64), np.floor(yi[inside] - 0.5).astype(np.int64)
    used = np.zeros((H, W), bool)
    for dy in (0, 1):
        for dx in (0, 1):
            yy, xx = yf + dy, np.clip(xf + dx, 0, W - 1)
            ok = yy < H if dy else np.ones_like(yy, bool)
            used[np.clip(yy[ok], 0, H - 1), xx[ok]] = True
    return int(used.sum())


def kernel_time(B, name, iters, dev):
    from ccvpe_b200 import models
    (H, W), (h, w), offset = SHAPES[name]
    mats = [models.rotate_matrix(a, (W, H)) for a in angles(B)]
    m = torch.tensor(mats, dtype=torch.float64, device=dev)
    xs = [torch.randint(0, 256, (B, H, W, 3), dtype=torch.uint8, device=dev) for _ in range(3)]
    outs = [torch.empty((B, 3, h, w), dtype=torch.uint8, device=dev) for _ in range(3)]
    for i in range(3):
        models.CVM_VIGOR.affine_u8(xs[i], m, (h, w), offset, out=outs[i])
    torch.cuda.synchronize()
    # the launches are captured in a CUDA graph, so the events time the kernels rather than the Python-side enqueue
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for i in range(iters):
            models.CVM_VIGOR.affine_u8(xs[i % 3], m, (h, w), offset, out=outs[i % 3])
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    graph.replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    read = 3 * sum(footprint_pixels(a, (H, W), (h, w), offset) for a in mats)
    nbytes = read + outs[0].numel()
    return {"B": B, "src": [H, W], "dst": [h, w], "offset": list(offset), "layout": "NHWC", "us_per_call": round(ms * 1e3, 1),
            "footprint_bytes": read, "output_bytes": outs[0].numel(), "gb_per_s": round(nbytes / ms / 1e6, 1),
            "share_of_hbm_peak": round(nbytes / ms / 1e6 / HBM_PEAK_GBS, 3)}


def host_pillow(n):
    from PIL import Image

    from ccvpe_b200 import models
    rng = np.random.default_rng(0)
    t = {}
    for name in SHAPES:
        (H, W), (h, w), (left, top) = SHAPES[name]
        ims = [Image.fromarray(rng.integers(0, 256, (H, W, 3), dtype=np.uint8)) for _ in range(n)]
        box = (left, top, left + w, top + h)
        ops = {"rotate": lambda im, a: im.rotate(a, Image.BILINEAR).crop(box) if left or top else
               im.rotate(a, Image.BILINEAR)}
        if left or top:
            ops["transform_to_box"] = lambda im, a: im.transform(
                (left + w, top + h), Image.AFFINE, models.rotate_matrix(a, (W, H)), Image.BILINEAR).crop(box)
        for op, f in ops.items():
            f(ims[0], 10.0)
            t0 = time.perf_counter()
            for im, a in zip(ims, angles(n)):
                f(im, a)
            t["%s_%s_ms" % (name, op)] = round((time.perf_counter() - t0) * 1e3 / n, 2)
    import PIL
    return dict(pillow=PIL.__version__, threads=1, cpu_count=os.cpu_count(), images=n, **t)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--iters", type=int, default=60, help="graph-captured launches per shape")
    ap.add_argument("--images", type=int, default=10, help="images transformed with Pillow on the host, per operation")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_affine.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    res = {"gpu": gpu_info(), "kernel": {name: kernel_time(args.batch, name, args.iters, dev) for name in SHAPES},
           "host": host_pillow(args.images)}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
