"""TEST INFRASTRUCTURE -- generates the model fixtures tests/golden/<config>.npz by running the UNMODIFIED reference.

    CCVPE_REFERENCE_ROOT=<checkout of tudelft-iv/CCVPE> python oracle/make_golden.py

For every configuration of BASELINE.json (class x ground shape x ori prior) the reference model is built
via `oracle/ref_shim.py`, its weights are overwritten by `ccvpe_b200.synthetic.fill_deterministic(seed)`, it is
run on `synthetic_pair(batch, shape, seed)` and, for each of the nine outputs (models.py:343), we store
  * the shape, the float64 sum and abs-sum of the whole tensor,
  * the values at 4096 fixed pseudo-random flat indices (all values if the tensor is smaller than 16384),
  * the host pose decode of train_VIGOR.py:290-326 (argmax index, row/col, cos/sin, angle).
The fixtures pin `oracle/ccvpe_oracle.py` (tests/test_oracle_golden.py); they are a few hundred kB each.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from ccvpe_b200.synthetic import GROUND_SHAPES, fill_deterministic, synthetic_pair  # noqa: E402
from oracle import ccvpe_oracle as orc  # noqa: E402
from oracle.ref_shim import load_reference_models  # noqa: E402

OUT_NAMES = ["logits", "heatmap", "ori", "scores1", "scores2", "scores3", "scores4", "scores5", "scores6"]
N_SAMPLES = 4096

#: name -> (variant, ground-shape key, ori_noise, circular_padding, batch, weight seed, input seed)
CONFIGS = {
    "vigor_fov360_b1": ("vigor", "vigor", None, True, 1, 3, 1),
    "vigor_fov360_b2": ("vigor", "vigor", None, True, 2, 4, 2),
    "vigor_prior72_fov180_b1": ("vigor_prior", "vigor_fov180", 72.0, False, 1, 5, 3),
    "vigor_prior72_fov108_b1": ("vigor_prior", "vigor_fov108", 72.0, False, 1, 6, 4),
    "vigor_prior180_fov360_b1": ("vigor_prior", "vigor", 180.0, True, 1, 7, 5),
    "kitti_b1": ("kitti", "kitti", None, None, 1, 8, 6),
    "oxford_b1": ("oxford", "oxford", None, None, 1, 9, 7),
}


def build_reference(ref_models, variant, ori_noise, circular):
    if variant == "vigor":
        return ref_models.CVM_VIGOR("cpu", circular)
    if variant == "vigor_prior":
        return ref_models.CVM_VIGOR_ori_prior("cpu", ori_noise, circular)
    if variant == "kitti":
        return ref_models.CVM_KITTI("cpu")
    return ref_models.CVM_OxfordRobotCar("cpu")


def sample_indices(numel: int, name: str) -> np.ndarray:
    if numel <= 4 * N_SAMPLES:
        return np.arange(numel, dtype=np.int64)
    rng = np.random.default_rng(numel)
    return np.sort(rng.choice(numel, N_SAMPLES, replace=False)).astype(np.int64)


def digest(outputs):
    rec = {}
    for name, t in zip(OUT_NAMES, outputs):
        a = t.detach().cpu().numpy()
        flat = a.reshape(-1)
        idx = sample_indices(flat.size, name)
        rec[name + ".shape"] = np.asarray(a.shape, np.int64)
        rec[name + ".sum"] = np.float64(flat.astype(np.float64).sum())
        rec[name + ".abssum"] = np.float64(np.abs(flat.astype(np.float64)).sum())
        rec[name + ".idx"] = idx
        rec[name + ".val"] = flat[idx].astype(np.float32)
    pose = orc.pose_decode(outputs[1].detach().numpy(), outputs[2].detach().numpy())
    for k, v in pose.items():
        rec["pose." + k] = v
    lg = outputs[0].detach()
    top = torch.topk(lg, 2, dim=1).values
    rec["logits.top2gap"] = (top[:, 0] - top[:, 1]).numpy().astype(np.float64)
    return rec


def main():
    torch.set_num_threads(8)  # fixtures were generated with 8 threads (reference is thread-count sensitive in the last bits)
    ref_models = load_reference_models()
    os.makedirs(os.path.join(ROOT, "tests", "golden"), exist_ok=True)
    for name, (variant, shape_key, noise, circular, batch, wseed, iseed) in CONFIGS.items():
        model = build_reference(ref_models, variant, noise, circular).eval()
        fill_deterministic(model.state_dict(), seed=wseed)
        grd, sat = synthetic_pair(batch, GROUND_SHAPES[shape_key], seed=iseed)
        with torch.no_grad():
            out = model(grd, sat)
        rec = digest(out)
        rec["meta"] = np.asarray([variant, shape_key, str(noise), str(circular), str(batch), str(wseed), str(iseed),
                                  torch.__version__])
        path = os.path.join(ROOT, "tests", "golden", name + ".npz")
        np.savez_compressed(path, **rec)
        print("%-28s -> %s (%.0f kB)  argmax %s  top2gap %s" % (name, os.path.relpath(path, ROOT),
              os.path.getsize(path) / 1e3, rec["pose.idx"].tolist(), rec["logits.top2gap"].tolist()))


if __name__ == "__main__":
    main()
