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


# ---------------------------------------------------------------------------------------------------------------------
# per-element bounds and guarded replays of the plan checks (tests/test_gpu_plan_parity.py, tests/test_gpu_encoder_plan.py)
# ---------------------------------------------------------------------------------------------------------------------
RHO_BF16 = 2.0 ** -8        # bound on the relative error of one bf16 store (its unit roundoff is 2^-9)
TINY = 2.0 ** -126          # smallest normal fp32 / bf16 magnitude


def subnormal_floor(t1):
    """Absolute allowance for flush-to-zero.  The tensor cores flush subnormal operands, products and partial sums: a term
    a*w of an output loses at most TINY * (|a| + |w| + 2) <= 2 TINY (|a| + 1)(|w| + 1); `t1` is that sum over the output's
    terms.  Without it, gradients that decay into the subnormal range (the orientation loss is a Gaussian blob, so its
    data gradients are ~1e-40 far from the blob) fail the relative bound although they are zero to within 1e-38.  The
    floor stays below 1e-30 for every shape here, far under any value the bound is meant to resolve."""
    return 2 * TINY * t1


def bound_check(got, ref, S, rho, tau, floor=0.0):
    """Returns (worst |got - ref| / (rho |ref| + tau S + floor), worst (|got - ref| - rho |ref| - floor) / S = the tau this
    tensor needs).  Where the bound is zero the element must be exact; a non-finite output where the reference is finite
    fails."""
    got, ref, S = got.to(torch.float64).reshape(-1), ref.to(torch.float64).reshape(-1), S.to(torch.float64).reshape(-1)
    if torch.is_tensor(floor):
        floor = floor.to(torch.float64).reshape(-1)
    d = (got - ref).abs()
    d = torch.where(torch.isfinite(d), d, torch.full_like(d, float("inf")))
    bound = rho * ref.abs() + tau * S + floor
    ratio = torch.where(bound > 0, d / bound.clamp_min(1e-300), torch.where(d > 0, float("inf"), 0.0))
    excess = (d - rho * ref.abs() - floor).clamp_min(0.0)
    need = torch.where(S > 0, excess / S.clamp_min(1e-300), torch.where(excess > 0, float("inf"), 0.0))
    return (float(ratio.max()) if ratio.numel() else 0.0), (float(need.max()) if need.numel() else 0.0)


def image_subset(B):
    """Images whose outputs are checked for the per-image operators: all of them up to 8, else 0, 1, B/2 and B-1."""
    return list(range(B)) if B <= 8 else sorted({0, 1, B // 2, B - 1})


SENTINEL = {torch.bfloat16: (torch.int16, -1), torch.float32: (torch.int32, -1)}    # all-ones bits: a NaN no kernel writes


def sentinel_bits(t):
    ity, _ = SENTINEL[t.dtype]
    return t.view(ity)


def guarded(n, dtype, guard, dev):
    """A sentinel-filled buffer of guard + n + guard elements; the output is buf[guard:guard + n]."""
    buf = torch.empty(guard + n + guard, dtype=dtype, device=dev)
    sentinel_bits(buf).fill_(SENTINEL[dtype][1])
    return buf


def guard_report(buf, n, guard, ref_out, written=None):
    """Problems of a replay into `guarded(n, ...)`: writes into the guards, output elements left unwritten, and output
    elements that differ from the plan's own output `ref_out`.  `written` (bool, shaped like ref_out): the elements the
    launch must write; the others must still hold the sentinel.  None = every element."""
    s = SENTINEL[buf.dtype][1]
    bits = sentinel_bits(buf)
    problems = []
    if not bool((bits[:guard] == s).all()):
        problems.append("wrote %d elements before the output" % int((bits[:guard] != s).sum()))
    if not bool((bits[guard + n:] == s).all()):
        problems.append("wrote %d elements past the output" % int((bits[guard + n:] != s).sum()))
    inner = bits[guard:guard + n]
    want = sentinel_bits(ref_out.reshape(-1))
    if written is not None:
        mask = written.reshape(-1)
        if not bool((inner[~mask] == s).all()):
            problems.append("wrote %d elements outside the ones it owns" % int((inner[~mask] != s).sum()))
        inner, want = inner[mask], want[mask]
    if bool((inner == s).any()):
        problems.append("left %d output elements unwritten" % int((inner == s).sum()))
    if not torch.equal(inner, want):
        problems.append("replay differs from the plan's output in %d elements" % int((inner != want).sum()))
    return problems


def guard_len(row):
    return (128 * row + 4096 + 511) // 512 * 512          # >= one 128-row tile; keeps the interior 1 KB aligned
