"""Shared test helpers (test infrastructure)."""
import numpy as np
import torch

from ccvpe_b200 import models as cvm
from ccvpe_b200.synthetic import GROUND_SHAPES, fill_deterministic, synthetic_pair

OUT_NAMES = ["logits", "heatmap", "ori", "scores1", "scores2", "scores3", "scores4", "scores5", "scores6"]

#: mirrors oracle/make_golden.py CONFIGS: name -> (variant, ground-shape key, ori_noise, circular, batch, wseed, iseed)
GOLDEN_CONFIGS = {
    "vigor_fov360_b1": ("vigor", "vigor", None, True, 1, 3, 1),
    "vigor_fov360_b2": ("vigor", "vigor", None, True, 2, 4, 2),
    "vigor_prior72_fov180_b1": ("vigor_prior", "vigor_fov180", 72.0, False, 1, 5, 3),
    "vigor_prior72_fov108_b1": ("vigor_prior", "vigor_fov108", 72.0, False, 1, 6, 4),
    "vigor_prior180_fov360_b1": ("vigor_prior", "vigor", 180.0, True, 1, 7, 5),
    "kitti_b1": ("kitti", "kitti", None, None, 1, 8, 6),
    "oxford_b1": ("oxford", "oxford", None, None, 1, 9, 7),
}
#: torch CPU threads of the run that generated the fixtures (oracle/make_golden.py): the CPU convolutions split their sums
#: by thread, so another count changes the last bits, which the unit orientation field amplifies to ~1e-3 where |v| ~ 0
GOLDEN_THREADS = 8


def build_model(variant, ori_noise, circular, wseed):
    if variant == "vigor":
        m = cvm.CVM_VIGOR("cpu", circular)
    elif variant == "vigor_prior":
        m = cvm.CVM_VIGOR_ori_prior("cpu", ori_noise, circular)
    elif variant == "kitti":
        m = cvm.CVM_KITTI("cpu")
    else:
        m = cvm.CVM_OxfordRobotCar("cpu")
    fill_deterministic(m.state_dict(), seed=wseed)
    return m.eval()


def config_inputs(name):
    variant, shape_key, noise, circular, batch, wseed, iseed = GOLDEN_CONFIGS[name]
    return synthetic_pair(batch, GROUND_SHAPES[shape_key], seed=iseed)


def oracle_forward(model, variant, noise, grd, sat, intermediates=None):
    from oracle import ccvpe_oracle as orc

    sd = {k: v.detach() for k, v in model.state_dict().items()}
    with torch.no_grad():
        return orc.forward_full(variant, sd, model.grd_efficientnet, model.sat_efficientnet, grd, sat, noise,
                                intermediates)


def ori_field_err(ori: torch.Tensor, ori_ref: torch.Tensor, ori_raw_ref: torch.Tensor) -> float:
    """Error of the unit orientation field measured on the field BEFORE normalisation: F.normalize divides by the
    per-pixel magnitude, so an absolute error d on the raw 2-vector v shows up as ~d/|v| on v/|v|.  Returns
    max_p |ori - ori_ref|_p * |v_p| / max|v|, i.e. the relative error of the raw field that explains the difference
    (equals the plain relative error wherever |v_p| is of the order of max|v|)."""
    mag = ori_raw_ref.detach().double().norm(dim=1, keepdim=True)
    d = (ori.detach().double().cpu() - ori_ref.detach().double()).abs()
    return (d * mag / ori_raw_ref.detach().double().abs().max()).max().item()


def rel_err(a: torch.Tensor, ref: torch.Tensor) -> float:
    """max |a - ref| / max |ref|  -- the tolerance measure used throughout (stated per test)."""
    a = a.detach().double().cpu()
    ref = ref.detach().double().cpu()
    denom = ref.abs().max().item()
    return (a - ref).abs().max().item() / (denom if denom > 0 else 1.0)


def check_against_golden(outputs, golden, tol, loose=None):
    """outputs: 9-tuple of tensors; golden: np.load of a tests/golden file."""
    worst = {}
    for name, t in zip(OUT_NAMES, outputs):
        a = t.detach().float().cpu().numpy()
        assert tuple(a.shape) == tuple(golden[name + ".shape"]), name
        flat = a.reshape(-1)
        ref = golden[name + ".val"]
        got = flat[golden[name + ".idx"]]
        scale = np.abs(ref).max()
        err = np.abs(got.astype(np.float64) - ref.astype(np.float64)).max() / (scale if scale > 0 else 1.0)
        worst[name] = err
        tol_n = (loose or {}).get(name, tol)
        assert err <= tol_n, "%s: sampled rel err %.3e > %.1e" % (name, err, tol)
        s_ref, as_ref = float(golden[name + ".sum"]), float(golden[name + ".abssum"])
        assert abs(flat.astype(np.float64).sum() - s_ref) <= tol * max(as_ref, 1e-30), name + " checksum"
    return worst
