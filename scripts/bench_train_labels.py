"""Dense vs compact training labels for the CVM_VIGOR training step.

Dense labels are the three maps per pair (gt, gt_with_ori [20, 512, 512], gt_orientation [2, 512, 512]) fed to
`losses.training_loss`; compact labels are (gt, bin_weights [20], ori_vec [2]) fed to `losses.training_loss_from_labels`.
Both give the same loss and gradients.  The two arms alternate within one run, so they see the same machine state.

  (a) loss stage: forward + backward of the loss alone on CVM_VIGOR B=8 bf16 outputs, CUDA events over --iters
      iterations per round (the 168 MB gt_with_ori of the dense arm does not fit the 126 MB L2)
  (b) end to end: one `training.GraphedTrainStep` per arm fed from pinned host buffers, double buffered as in
      bench_train.py (images + labels copied every step); pairs/s, H2D bytes per step and the copy time of one step's
      inputs alone.  Under torchrun: one process per GPU, 8 pairs each (weak scaling), bucketed gradient all-reduce.
  (c) host cost per pair of building the labels on one CPU core: the dense maps vs gt + orientation_labels.

    python scripts/bench_train_labels.py --out DIR            # one GPU
    torchrun --nproc-per-node 8 scripts/bench_train_labels.py --out DIR --skip-loss --skip-host

Writes DIR/r05_train_labels[_nN].json and prints a summary.  Needs a CUDA device.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from ccvpe_b200 import losses, models  # noqa: E402
from ccvpe_b200.ddp import GradientAllReducer  # noqa: E402
from ccvpe_b200.synthetic import fill_deterministic, synthetic_ground_truth, synthetic_labels, synthetic_pair  # noqa: E402
from ccvpe_b200.training import GraphedTrainStep  # noqa: E402

GROUND = (320, 640)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[int(os.environ.get("LOCAL_RANK", "0"))] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def nbytes(ts):
    return sum(t.numel() * t.element_size() for t in ts)


def dense_labels(B, seed):
    return list(synthetic_ground_truth(B, seed=seed))


def compact_labels(B, seed):
    gt, angles = synthetic_labels(B, seed=seed)
    return [gt, *losses.orientation_labels(angles)]


def loss_stage(model, B, dev, rounds, iters):
    grd, sat = (t.to(dev) for t in synthetic_pair(B, GROUND, seed=5))
    with torch.no_grad():
        out = model(grd, sat)
    leaves = [t.detach().clone().requires_grad_(i != 1) for i, t in enumerate(out)]
    wrt = [leaves[0], leaves[2]] + leaves[3:9]
    dense = [t.to(dev) for t in dense_labels(B, 1)]
    compact = [t.to(dev) for t in compact_labels(B, 1)]
    arms = {"dense": lambda: losses.training_loss(leaves, *dense), "compact": lambda: losses.training_loss_from_labels(leaves, *compact)}
    vals = {}
    for name, f in arms.items():
        for _ in range(5):
            torch.autograd.grad(f(), wrt)
        loss = f()
        vals[name] = (float(loss), [g.float().sum().item() for g in torch.autograd.grad(loss, wrt)])
    same = vals["dense"] == vals["compact"]
    ms = {k: [] for k in arms}
    for _ in range(rounds):
        for name, f in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(iters):
                torch.autograd.grad(f(), wrt)
            e1.record()
            torch.cuda.synchronize()
            ms[name].append(e0.elapsed_time(e1) / iters)
    res = {k: {"ms_median": round(statistics.median(v), 4), "ms_min": round(min(v), 4), "ms_max": round(max(v), 4)}
           for k, v in ms.items()}
    res.update(batch=B, precision="bf16", rounds=rounds, iters_per_round=iters, identical_loss_and_grad_sums=same,
               label_bytes_on_device={"dense": nbytes(dense), "compact": nbytes(compact)},
               note="forward + backward (torch.autograd.grad) of the loss alone on fixed CVM_VIGOR outputs; median over "
                    "rounds of the mean per iteration; the arms alternate every round")
    return res


def e2e(model, B, dev, rank, world, rounds, steps):
    reducer = GradientAllReducer(model)
    opt = torch.optim.Adam([p for p in model.parameters() if p.requires_grad], lr=1e-4, betas=(0.9, 0.999), fused=True,
                           capturable=True)
    torch.backends.cudnn.benchmark = True

    def make(loss_fn):
        def step(grd, sat, *labels):
            reducer.zero_grad()
            loss = loss_fn(model(grd, sat), *labels)
            loss.backward()
            reducer.finish()
            opt.step()
            return loss.detach()
        return step

    imgs = list(synthetic_pair(B, GROUND, seed=200 + rank))
    arms = {}
    for name, labels, fn in (("dense", dense_labels(B, 200 + rank), losses.training_loss),
                             ("compact", compact_labels(B, 200 + rank), losses.training_loss_from_labels)):
        host = [t.pin_memory() for t in imgs + labels]
        resident = [t.to(dev) for t in host]
        resident[0] = resident[0].contiguous(memory_format=torch.channels_last)
        resident[1] = resident[1].contiguous(memory_format=torch.channels_last)
        step = make(fn)
        for _ in range(2):
            step(*resident)
        graph = GraphedTrainStep(step, resident, warmup=2)
        arms[name] = dict(host=host, graph=graph, dev_in=[[torch.empty_like(t) for t in graph.static_in] for _ in range(2)])
    copy_stream = torch.cuda.Stream(device=dev)
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()

    def run(arm, n):
        host, graph, dev_in = arm["host"], arm["graph"], arm["dev_in"]
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

        nxt = upload(0)
        for i in range(n):
            slot = i % 2
            ev = nxt
            if i + 1 < n:
                nxt = upload(1 - slot)
            torch.cuda.current_stream().wait_event(ev)
            loss = graph(*dev_in[slot])
            slot_free[slot] = torch.cuda.Event()
            slot_free[slot].record()
            loss_host.copy_(loss, non_blocking=True)
            done = torch.cuda.Event()
            done.record()
            done.synchronize()
        return float(loss_host)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    for arm in arms.values():
        run(arm, 3)
    ms = {k: [] for k in arms}
    for _ in range(rounds):
        for name, arm in arms.items():
            barrier()
            t0 = time.perf_counter()
            run(arm, steps)
            barrier()
            ms[name].append((time.perf_counter() - t0) * 1e3 / steps)
    copy_ms = {}
    for name, arm in arms.items():                     # the copy of one step's inputs alone, nothing else running
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        c0.record()
        for _ in range(10):
            for d, h in zip(arm["dev_in"][0], arm["host"]):
                d.copy_(h, non_blocking=True)
        c1.record()
        torch.cuda.synchronize()
        copy_ms[name] = c0.elapsed_time(c1) / 10
    if world > 1:
        t = torch.tensor([statistics.median(ms["dense"]), statistics.median(ms["compact"])], dtype=torch.float64, device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        med = dict(zip(("dense", "compact"), t.tolist()))
    else:
        med = {k: statistics.median(v) for k, v in ms.items()}
    res = {}
    for name, arm in arms.items():
        h2d = nbytes(arm["host"])
        res[name] = {"pairs_per_s": round(world * B / (med[name] / 1e3), 2), "ms_per_step_median": round(med[name], 3),
                     "ms_per_step_rounds_rank0": [round(v, 3) for v in ms[name]], "h2d_bytes_per_step": h2d,
                     "h2d_copy_alone_ms_rank0": round(copy_ms[name], 3),
                     "h2d_copy_alone_gbs_rank0": round(h2d / (copy_ms[name] * 1e-3) / 1e9, 1)}
    res.update(world=world, batch_per_gpu=B, rounds=rounds, steps_per_round=steps, precision="bf16",
               note="GraphedTrainStep (whole step in one CUDA graph) fed from pinned host buffers, double buffered; every step "
                    "copies images + labels and reads the loss back; host wall clock over the round, max over ranks")
    return res


def host_cost(B, reps):
    torch.set_num_threads(1)
    arms = {"dense": lambda s: synthetic_ground_truth(B, seed=s),
            "compact": lambda s: (lambda gt, a: (gt, losses.orientation_labels(a)))(*synthetic_labels(B, seed=s))}
    ms = {k: [] for k in arms}
    for r in range(reps):
        for name, f in arms.items():
            t0 = time.perf_counter()
            f(r)
            ms[name].append((time.perf_counter() - t0) * 1e3 / B)
    return {k: {"ms_per_pair_median": round(statistics.median(v), 3), "ms_per_pair_min": round(min(v), 3)} for k, v in ms.items()} | {
        "batch": B, "reps": reps, "threads": 1, "host_cores": os.cpu_count(),
        "note": "synthetic_ground_truth (the Gaussian and the dense maps) vs synthetic_labels + orientation_labels, one "
                "torch thread; both include drawing the Gaussian"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for the JSON result")
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--loss-rounds", type=int, default=6)
    ap.add_argument("--loss-iters", type=int, default=50)
    ap.add_argument("--e2e-rounds", type=int, default=4)
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--host-reps", type=int, default=5)
    ap.add_argument("--skip-loss", action="store_true")
    ap.add_argument("--skip-host", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_train_labels.py needs a CUDA device")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=dev)
    model = models.CVM_VIGOR("cuda", True)
    fill_deterministic(model.state_dict(), seed=0)
    model = model.to(dev).set_precision("bf16").train()
    res = {"card": card(), "torch": torch.__version__}
    if rank == 0 and not args.skip_loss:
        res["a_loss_stage"] = loss_stage(model, args.batch, dev, args.loss_rounds, args.loss_iters)
    res["b_end_to_end"] = e2e(model, args.batch, dev, rank, world, args.e2e_rounds, args.e2e_steps)
    if rank == 0 and not args.skip_host:
        res["c_host_cost"] = host_cost(args.batch, args.host_reps)
    if rank == 0:
        os.makedirs(args.out, exist_ok=True)
        path = os.path.join(args.out, "r05_train_labels%s.json" % ("_n%d" % world if world > 1 else ""))
        with open(path, "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps(res, indent=1), flush=True)
    if world > 1:
        torch.cuda.synchronize()
        torch.distributed.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        os._exit(0)                     # the captured graphs hold NCCL work: leave without the process-group destructor


if __name__ == "__main__":
    main()
