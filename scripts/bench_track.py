"""Sequential location filter (decoder.track_step / ccvpe_track_step): kernel time, bandwidth, and its cost per frame next to
the bf16 Oxford RobotCar model at batch 1.

1. `track_step` alone, 512x512 maps, B in {1, 64}, sigma in {0, 2, 8, 32} pixels, epsilon 1e-3, a rotation + sub-pixel
   shift motion.  Each arm's `--iters` steps are captured in one CUDA graph, so the events time the kernels rather than the
   Python-side enqueue; the steps cycle through 4 copies of (belief, heatmap, motion): 512 MiB at B = 64, four times the
   126 MB L2, so every step reads its inputs from HBM (at B = 1 the 8 MiB stay in L2, and the floor is the latency of the
   three launches).  Arms are timed in turn for `--reps` rounds; each reports the median and the spread.  GB/s and the
   share of the 7.7 TB/s data-sheet HBM bandwidth are given for two byte counts: the minimal traffic (12 B per pixel: read
   belief and heatmap, write belief) and the traffic of the three launches (warp + row blur: read belief, write the
   scratch plane; column blur: read the scratch plane with each tile's halo rows, read heatmap, write q; normalise: read
   q, write belief).
2. Per-frame latency of bf16 CVM_OxfordRobotCar in CUDA-graph mode at batch 1: forward + decode_pose against forward +
   track_step + decode_pose, each frame ending in a host read of the decoded pixel as a sequential loop does.

Prints one JSON object (with the GPU's name and power limit); `--out FILE` also writes it there."""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

COPIES = 4
SIGMAS = (0.0, 2.0, 8.0, 32.0)
BATCHES = (1, 64)
EPS = 1e-3
HBM_BYTES_PER_S = 7.7e12     # NVIDIA HGX B200 data sheet, one GPU
SIZE = 512


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as exc:                                    # noqa: BLE001 -- reported, not fatal
        return {"name": torch.cuda.get_device_name(0), "nvidia_smi": "unavailable (%s)" % exc}


def design_bytes(B, H, W, sigma):
    """Bytes the three launches move (the tile geometry of track.cu: 32 x 64 output tiles, r halo rows each side)."""
    r = math.ceil(3 * sigma)
    staged = sum(min(i0 + 64 + r, H) - max(i0 - r, 0) for i0 in range(0, H, 64))   # rows of the scratch plane per column
    plane = B * H * W * 4
    return plane * 2 + B * staged * W * 4 + plane * 2 + plane * 2


def motion_matrix():
    from ccvpe_b200.models import rotate_matrix, track_motion

    prev = rotate_matrix(10.0, (SIZE, SIZE))
    new = rotate_matrix(12.5, (SIZE, SIZE))
    new[2] += 3.3
    new[5] -= 1.7
    return track_motion(prev, new, (0.25, -0.75))


def time_track(B, iters, reps, dev):
    from ccvpe_b200 import cabi
    from ccvpe_b200.synthetic import synthetic_mixture

    beliefs = [synthetic_mixture(B, 8, SIZE, SIZE, seed=10 + c).to(dev) for c in range(COPIES)]
    heats = [(synthetic_mixture(B, 8, SIZE, SIZE, seed=20 + c) + 1e-7).to(dev) for c in range(COPIES)]
    motions = [torch.tensor([motion_matrix()] * B, dtype=torch.float64, device=dev) for _ in range(COPIES)]
    ev = torch.empty(B, dtype=torch.float64, device=dev)
    rs = torch.empty(B, dtype=torch.uint8, device=dev)
    scratch = torch.empty(cabi.track_scratch_bytes(B, SIZE, SIZE), dtype=torch.uint8, device=dev)
    graphs = {}
    for sigma in SIGMAS:
        for c in range(COPIES):
            cabi.track_step(beliefs[c], heats[c], motions[c], sigma, EPS, ev, rs, scratch)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for i in range(iters):
                c = i % COPIES
                cabi.track_step(beliefs[c], heats[c], motions[c], sigma, EPS, ev, rs, scratch)
        g.replay()
        graphs[sigma] = g
    torch.cuda.synchronize()
    samples = {s: [] for s in SIGMAS}
    for _ in range(reps):
        for sigma, g in graphs.items():                         # arms alternate within every round
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            samples[sigma].append(e0.elapsed_time(e1) * 1e3 / iters)
    assert not rs.any(), "a timed step reset"
    minimal = B * SIZE * SIZE * 12
    res = {}
    for sigma in SIGMAS:
        us = sorted(samples[sigma])
        med = us[len(us) // 2]
        actual = design_bytes(B, SIZE, SIZE, sigma)
        res["sigma=%g" % sigma] = {
            "us_median": round(med, 2), "us_min": round(us[0], 2), "us_max": round(us[-1], 2),
            "minimal_bytes": minimal, "minimal_gb_per_s": round(minimal / med / 1e3, 1),
            "minimal_share_of_hbm_bound": round(minimal / HBM_BYTES_PER_S / (med * 1e-6), 3),
            "design_bytes": actual, "design_gb_per_s": round(actual / med / 1e3, 1),
            "design_share_of_hbm_bound": round(actual / HBM_BYTES_PER_S / (med * 1e-6), 3)}
    return res


def time_oxford(frames, reps, dev):
    from ccvpe_b200 import models
    from ccvpe_b200.synthetic import GROUND_SHAPES, fill_deterministic, synthetic_pair

    model = models.CVM_OxfordRobotCar(dev).eval()
    fill_deterministic(model.state_dict(), seed=0)
    model = model.to(dev).set_precision("bf16")
    model.set_cuda_graph(True)
    grd, sat = (t.to(dev) for t in synthetic_pair(1, GROUND_SHAPES["oxford"], seed=1))
    motion = torch.tensor([motion_matrix()], dtype=torch.float64, device=dev)
    belief = None

    def plain():
        out = model(grd, sat)
        return model.decode_pose(out[1], out[2])

    def tracked():
        nonlocal belief
        out = model(grd, sat)
        if belief is None:
            belief = out[1].clone()
        model.track_step(belief, out[1], motion, 2.0, EPS)
        return model.decode_pose(belief, out[2])

    arms = {"forward+decode_pose": plain, "forward+track_step+decode_pose": tracked}
    with torch.no_grad():
        for fn in arms.values():
            for _ in range(5):
                fn()["idx"].cpu()
        torch.cuda.synchronize()
        samples = {k: [] for k in arms}
        for _ in range(reps):
            for name, fn in arms.items():
                t0 = time.perf_counter()
                for _ in range(frames):
                    fn()["idx"].cpu()                         # a sequential loop reads every frame's answer
                samples[name].append((time.perf_counter() - t0) / frames * 1e3)
    res = {}
    for name, ms in samples.items():
        ms = sorted(ms)
        res[name] = {"ms_per_frame_median": round(ms[len(ms) // 2], 4), "ms_min": round(ms[0], 4),
                     "ms_max": round(ms[-1], 4)}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=40)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--frames", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_track needs a CUDA device")
    dev = torch.device("cuda:0")
    result = {"gpu": gpu_info(), "map": [SIZE, SIZE], "epsilon": EPS, "iters": a.iters, "reps": a.reps,
              "copies_cycled": COPIES, "hbm_bound_bytes_per_s": HBM_BYTES_PER_S}
    for B in BATCHES:
        result["track_step B=%d" % B] = time_track(B, a.iters, a.reps, dev)
    result["oxford_b1_bf16_graph"] = time_oxford(a.frames, a.reps, dev)
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
