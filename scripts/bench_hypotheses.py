"""Pose hypotheses (decoder.decode_hypotheses / ccvpe_pose_hypotheses) against the argmax decode (decode_pose) it extends.

B = 64 pairs of 512x512 heatmaps, two inputs:
  * "model": the heatmaps and orientation fields of bf16 CVM_VIGOR with seeded weights on synthetic images;
  * "mixture8": 8-Gaussian mixtures (synthetic.synthetic_mixture), with the model run's orientation fields.
Arms: decode_pose, and decode_hypotheses with k in {1, 8, 32} x radius in {4, 16, 64} pixels.  Each arm's `--iters`
launches are captured in one CUDA graph, so the events time the kernels rather than the Python-side enqueue; the launches
cycle through 4 copies of the heatmaps (256 MiB, twice the 126 MB L2), so every pass reads its maps from HBM.  The arms
are timed in turn, `--reps` rounds, and each arm reports the median and the spread over the rounds.  GB/s counts the
heatmap bytes read once (B * 512 * 512 * 4), the traffic both decodes need at least.

Prints one JSON object (with the GPU's name and power limit); `--out FILE` also writes it there."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

COPIES = 4
KS = (1, 8, 32)
RADII = (4, 16, 64)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as exc:                                    # noqa: BLE001 -- reported, not fatal
        return {"name": torch.cuda.get_device_name(0), "nvidia_smi": "unavailable (%s)" % exc}


def model_outputs(B, dev):
    from ccvpe_b200 import models
    from ccvpe_b200.synthetic import GROUND_SHAPES, fill_deterministic, synthetic_pair

    model = models.CVM_VIGOR("cuda", True).eval()
    fill_deterministic(model.state_dict(), seed=0)
    model = model.to(dev).set_precision("bf16")
    heats, ori = [], None
    for c in range(COPIES):
        grd, sat = synthetic_pair(B, GROUND_SHAPES["vigor"], seed=c)
        with torch.no_grad():
            out = model(grd.to(dev), sat.to(dev))
        heats.append(out[1].contiguous())
        ori = out[2].contiguous() if ori is None else ori
    del model
    return heats, ori


def arms(B, dev):
    """name -> (launch(heatmap, ori), outputs) with preallocated outputs"""
    from ccvpe_b200 import cabi

    out = {}
    p = dict(idx=torch.empty(B, dtype=torch.int64, device=dev), rc=torch.empty(B, 2, dtype=torch.int32, device=dev),
             cs=torch.empty(B, 2, device=dev), angle=torch.empty(B, dtype=torch.float64, device=dev),
             valid=torch.empty(B, dtype=torch.uint8, device=dev),
             scratch=torch.empty(cabi.pose_scratch_bytes(B, 512 * 512), dtype=torch.uint8, device=dev))
    out["decode_pose"] = (lambda h, o, p=p: cabi.pose_decode(h, o, p["idx"], p["rc"], p["cs"], p["angle"], p["valid"],
                                                             p["scratch"]), p)
    for k in KS:
        for r in RADII:
            q = dict(idx=torch.empty(B, k, dtype=torch.int64, device=dev),
                     rc=torch.empty(B, k, 2, dtype=torch.int32, device=dev), value=torch.empty(B, k, device=dev),
                     mass=torch.empty(B, k, device=dev), cs=torch.empty(B, k, 2, device=dev),
                     angle=torch.empty(B, k, dtype=torch.float64, device=dev),
                     valid=torch.empty(B, k, dtype=torch.uint8, device=dev),
                     count=torch.empty(B, dtype=torch.int32, device=dev))
            out["hypotheses k=%d r=%d" % (k, r)] = (
                lambda h, o, k=k, r=r, q=q: cabi.pose_hypotheses(h, o, k, r, q["idx"], q["rc"], q["value"], q["mass"],
                                                                 q["cs"], q["angle"], q["valid"], q["count"]), q)
    return out


def time_input(heats, ori, B, iters, reps):
    table = arms(B, heats[0].device)
    graphs = {}
    for name, (launch, _) in table.items():
        for h in heats:
            launch(h, ori)                                      # warm-up, and the function attributes, outside capture
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for i in range(iters):
                launch(heats[i % len(heats)], ori)
        g.replay()
        graphs[name] = g
    torch.cuda.synchronize()
    samples = {name: [] for name in table}
    for _ in range(reps):
        for name, g in graphs.items():                          # arms alternate within every round
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            samples[name].append(e0.elapsed_time(e1) * 1e3 / iters)
    nbytes = B * 512 * 512 * 4
    res = {}
    for name, (launch, outs) in table.items():
        us = sorted(samples[name])
        med = us[len(us) // 2]
        row = {"us_median": round(med, 1), "us_min": round(us[0], 1), "us_max": round(us[-1], 1),
               "heatmap_gb_per_s": round(nbytes / med / 1e3, 1)}
        launch(heats[0], ori)
        torch.cuda.synchronize()
        if "count" in outs:
            row["mean_count"] = round(float(outs["count"].float().mean()), 2)
            row["mean_mass0"] = round(float(outs["mass"][:, 0].double().mean()), 4)
        res[name] = row
    # the first hypothesis is the argmax: checked on the data just timed
    _, pose = table["decode_pose"]
    for k in KS:
        hyp = table["hypotheses k=%d r=4" % k][1]
        assert torch.equal(hyp["idx"][:, 0], pose["idx"]), "hypothesis 0 differs from decode_pose"
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--iters", type=int, default=40)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_hypotheses needs a CUDA device")
    from ccvpe_b200.synthetic import synthetic_mixture

    dev = torch.device("cuda:0")
    heats, ori = model_outputs(a.batch, dev)
    result = {"gpu": gpu_info(), "batch": a.batch, "map": [512, 512], "iters": a.iters, "reps": a.reps,
              "heatmap_bytes": a.batch * 512 * 512 * 4, "copies_cycled": COPIES}
    result["model"] = time_input(heats, ori, a.batch, a.iters, a.reps)
    mix = [synthetic_mixture(a.batch, 8, seed=c).to(dev) for c in range(COPIES)]
    result["mixture8"] = time_input(mix, ori, a.batch, a.iters, a.reps)
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
