"""Training from poses: `ccvpe_pose_labels` builds a pair's location label, its pooled pyramid, its orientation bin weights
and its orientation vector on the device from (row, col, angle).

CPU: the binding and the C entry point refuse bad arguments before any launch, and `synthetic_poses` draws what
`synthetic_labels` draws.  GPU, every comparison exact: gt against NumPy float64 rounded once to float32, the pyramid
against `gt_pyramid` and `F.max_pool2d`, the bin weights and vector against `losses.orientation_labels` bit for bit, the
loss and gradients against `training_loss_from_labels` fed host-built labels, and a CUDA graph that redraws the
augmentation matrices and poses in place against eager steps."""
import ctypes
import math

import numpy as np
import pytest
import torch
from torch.nn import functional as F

from ccvpe_b200 import cabi, losses, models
from ccvpe_b200.synthetic import GROUND_SHAPES, synthetic_labels, synthetic_pair, synthetic_poses
from helpers import build_model

KS = (64, 32, 16, 8, 4, 2)
NAN = float("nan")
INF = float("inf")


def _np_gt(poses, H, W, sigma):
    """The reference location label: NumPy float64, rounded once to float32."""
    ys = np.arange(H, dtype=np.float64)[:, None]
    xs = np.arange(W, dtype=np.float64)[None, :]
    out = np.empty((len(poses), 1, H, W), dtype=np.float32)
    with np.errstate(all="ignore"):
        for b, (row, col, _angle) in enumerate(poses):
            out[b, 0] = np.exp(-(((ys - row) ** 2 + (xs - col) ** 2) / (2.0 * sigma ** 2))).astype(np.float32)
    return torch.from_numpy(out)


def _np_gt_f64(row, col, i, j, sigma):
    return math.exp(-(((i - row) ** 2 + (j - col) ** 2) / (2.0 * sigma ** 2)))


def _assert_same_floats(got, want, what, poses=None, sigma=None):
    """Equal values, NaN where the reference has NaN.  A failure lists the differing elements with the float64 value
    both sides rounded, so a last-bit disagreement of the two float64 `exp` at a float32 rounding boundary shows as such."""
    got, want = got.cpu(), want.cpu()
    assert got.shape == want.shape and got.dtype == want.dtype, (what, got.shape, want.shape)
    nan = torch.isnan(want)
    assert torch.equal(torch.isnan(got), nan), "%s: NaN positions differ" % what
    diff = (got != want) & ~nan
    if bool(diff.any()):
        lines = []
        for idx in diff.nonzero()[:10].tolist():
            line = "%s got %r want %r" % (idx, float(got[tuple(idx)]), float(want[tuple(idx)]))
            if poses is not None:
                b, _, i, j = idx
                line += " float64 %r" % _np_gt_f64(poses[b][0], poses[b][1], i, j, sigma)
            lines.append(line)
        raise AssertionError("%s: %d of %d elements differ\n%s" % (what, int(diff.sum()), want.numel(), "\n".join(lines)))


# ---------------------------------------------------------------------------------------------------------------
# CPU: argument checks before any launch
# ---------------------------------------------------------------------------------------------------------------
def _args(B=2, H=128, W=192, n_bins=20):
    return dict(poses=torch.zeros(B, 3, dtype=torch.float64), sigma=4.0, n_bins=n_bins, gt=torch.zeros(B, 1, H, W),
                pyramid=torch.zeros(cabi.gt_pyramid_elems(B, H, W)), bin_weights=torch.zeros(B, n_bins),
                ori_vec=torch.zeros(B, 2))


def _call(**kw):
    a = _args()
    a.update(kw)
    cabi.pose_labels(a["poses"], a["sigma"], a["n_bins"], a["gt"], a["pyramid"], a["bin_weights"], a["ori_vec"])


@pytest.mark.parametrize("kw,msg", [
    (dict(poses=torch.zeros(2, 3)), "poses must be a contiguous float64"),
    (dict(poses=torch.zeros(2, 4, dtype=torch.float64)), "poses must be a contiguous float64"),
    (dict(poses=torch.zeros(6, dtype=torch.float64)), "poses must be a contiguous float64"),
    (dict(poses=torch.zeros(0, 3, dtype=torch.float64)), "poses must be a contiguous float64"),
    (dict(poses=torch.zeros(3, 2, dtype=torch.float64).t()), "poses must be a contiguous float64"),
    (dict(gt=torch.zeros(2, 1, 128, 192, dtype=torch.float64)), "gt must be a float32"),
    (dict(gt=torch.zeros(3, 1, 128, 192)), "gt must have shape"),
    (dict(gt=torch.zeros(2, 128, 192)), "gt must have shape"),
    (dict(gt=torch.zeros(2, 1, 192, 128).transpose(2, 3)), "gt must be contiguous"),
    (dict(gt=torch.zeros(2, 1, 96, 192)), "multiples of 64"),
    (dict(gt=torch.zeros(2, 1, 128, 200)), "multiples of 64"),
    (dict(pyramid=torch.zeros(cabi.gt_pyramid_elems(2, 128, 192) - 1)), "pyramid must have shape"),
    (dict(pyramid=torch.zeros(cabi.gt_pyramid_elems(2, 128, 192)).half()), "pyramid must be a float32"),
    (dict(bin_weights=torch.zeros(2, 16)), "bin_weights must have shape"),
    (dict(bin_weights=torch.zeros(20, 2).t()), "bin_weights must be contiguous"),
    (dict(bin_weights=torch.zeros(2, 20, dtype=torch.bfloat16)), "bin_weights must be a float32"),
    (dict(ori_vec=torch.zeros(2, 3)), "ori_vec must have shape"),
    (dict(ori_vec=torch.zeros(2, 2, dtype=torch.float64)), "ori_vec must be a float32"),
    (dict(ori_vec=torch.zeros(2, 2).t()), "ori_vec must be contiguous"),
    (dict(sigma=0.0), "sigma"), (dict(sigma=-4.0), "sigma"), (dict(sigma=INF), "sigma"), (dict(sigma=NAN), "sigma"),
    (dict(sigma=True), "sigma"), (dict(sigma="4"), "sigma"),
    (dict(n_bins=9, bin_weights=torch.zeros(2, 9)), "n_bins"), (dict(n_bins=33, bin_weights=torch.zeros(2, 33)), "n_bins"),
    (dict(n_bins=20.0), "n_bins"),
    ({}, "CUDA"),                                # well-formed CPU tensors: refused for the device, never launched
])
def test_pose_labels_binding_refuses_bad_arguments(kw, msg):
    with pytest.raises(cabi.CcvpeError, match=msg):
        _call(**kw)


def test_labels_from_poses_refuses_bad_arguments():
    cpu = torch.zeros(2, 3, dtype=torch.float64)
    with pytest.raises(cabi.CcvpeError, match="CUDA"):
        losses.labels_from_poses(cpu)
    with pytest.raises(cabi.CcvpeError, match="CUDA"):
        losses.training_loss_from_poses(_outputs(2, 20), cpu)


def _outputs(B, n_bins, odd_level=None):
    outputs = [torch.zeros(B, 512 * 512), torch.zeros(B, 1, 512, 512), torch.zeros(B, 2, 512, 512)]
    outputs += [torch.zeros(B, 9 if level == odd_level else n_bins, 512 // k, 512 // k) for level, k in enumerate(KS, 1)]
    return outputs


def test_training_loss_from_poses_refuses_mismatched_bins():
    """CVM_VIGOR_ori_prior's levels carry 2k+1 orientation channels: refused before any launch, naming the level (9
    channels everywhere is refused as an n_bins outside [10, 32])."""
    poses = torch.zeros(1, 3, dtype=torch.float64)
    with pytest.raises(cabi.CcvpeError, match="score volume 3 has shape"):
        losses.training_loss_from_poses(_outputs(1, 20, odd_level=3), poses)
    with pytest.raises(cabi.CcvpeError, match="n_bins"):
        losses.training_loss_from_poses(_outputs(1, 9), poses)


def test_c_abi_refuses_bad_arguments_before_launch():
    """The C entry point checks its arguments itself (the pointers below are never dereferenced)."""
    lib = cabi.load()
    p = ctypes.c_void_p(4096)
    bad = -1                                                                    # CCVPE_ERR_BAD_ARGUMENT

    def call(poses=p, B=1, H=64, W=64, sigma=4.0, n_bins=20, gt=p, pyr=p, w=p, v=p):
        return lib.ccvpe_pose_labels(poses, B, H, W, sigma, n_bins, gt, pyr, w, v, None)

    for B, H, W in [(1, 100, 128), (1, 128, 96), (2, 0, 64), (0, 64, 64), (1, -64, 64), (70000, 64, 64)]:
        assert call(B=B, H=H, W=W) == bad, (B, H, W)
        assert b"multiples of 64" in lib.ccvpe_last_error()
    for kw in (dict(poses=None), dict(gt=None), dict(pyr=None), dict(w=None), dict(v=None)):
        assert call(**kw) == bad, kw
        assert b"null pointer" in lib.ccvpe_last_error()
    for kw in (dict(gt=ctypes.c_void_p(4100)), dict(poses=ctypes.c_void_p(4100)), dict(pyr=ctypes.c_void_p(4098)),
               dict(w=ctypes.c_void_p(4097)), dict(v=ctypes.c_void_p(4099))):
        assert call(**kw) == bad, kw
        assert b"misaligned" in lib.ccvpe_last_error()
    for sigma in (0.0, -1.0, INF, -INF, NAN):
        assert call(sigma=sigma) == bad, sigma
        assert b"sigma" in lib.ccvpe_last_error()
    for n_bins in (9, 33, 0, -20):
        assert call(n_bins=n_bins) == bad, n_bins
        assert b"n_bins" in lib.ccvpe_last_error()


def _draws_before(batch, seed, size):
    """The random sequence synthetic_labels has always drawn, verbatim."""
    g = torch.Generator().manual_seed(20_000 + seed)
    out = []
    for _ in range(batch):
        cy, cx = (torch.rand(2, generator=g) * (size - 64) + 32).tolist()
        out.append((cy, cx, float(torch.rand(1, generator=g)) * 360.0))
    return out


@pytest.mark.parametrize("batch,seed,size", [(1, 0, 512), (5, 3, 512), (4, 7, 128), (3, 11, 64), (8, 200, 512)])
def test_synthetic_poses_are_synthetic_labels_draws(batch, seed, size):
    poses = synthetic_poses(batch, seed=seed, size=size)
    assert poses.dtype == torch.float64 and poses.shape == (batch, 3) and not poses.is_cuda
    assert poses.tolist() == [list(d) for d in _draws_before(batch, seed, size)]
    gt, angles = synthetic_labels(batch, seed=seed, size=size)
    assert torch.equal(angles, poses[:, 2])
    ys = torch.arange(size, dtype=torch.float32).view(size, 1)
    xs = torch.arange(size, dtype=torch.float32).view(1, size)
    for b, (cy, cx, _) in enumerate(poses.tolist()):
        assert torch.equal(gt[b, 0], torch.exp(-((ys - cy) ** 2 + (xs - cx) ** 2) / (2.0 * 4.0 ** 2)))
    assert float(angles.min()) >= 0.0 and float(angles.max()) < 360.0


# ---------------------------------------------------------------------------------------------------------------
# GPU: gt and its pyramid
# ---------------------------------------------------------------------------------------------------------------
_SPECIAL_128x192 = [                        # (row, col) on a 128 x 192 map
    (64.0, 96.0), (10.0, 100.0),                               # integer
    (10.25, 100.7), (77.123456789, 3.0000001),                 # fractional
    (0.0, 0.0), (127.0, 191.0), (-0.5, 191.5), (127.9, -0.3),  # corners
    (-30.0, 50.0), (500.0, -100.0), (-1e6, 1e6), (1e300, 5.0),  # outside the map, the last one overflowing to inf
    (NAN, 20.0), (20.0, NAN), (INF, 5.0), (-INF, -INF),         # non-finite centres
]


def _labels_into_guarded(poses, H, W, sigma, n_bins, dev):
    """cabi.pose_labels into views inside sentinel-filled buffers: returns the outputs and a check that no guard changed."""
    B = poses.shape[0]
    guard, sentinel = 4096, -1234.5
    sizes = {"gt": B * H * W, "pyramid": cabi.gt_pyramid_elems(B, H, W), "bin_weights": B * n_bins, "ori_vec": 2 * B}
    bufs = {k: torch.full((n + 2 * guard,), sentinel, device=dev) for k, n in sizes.items()}
    views = {k: bufs[k][guard:guard + n] for k, n in sizes.items()}
    gt, w, v = views["gt"].view(B, 1, H, W), views["bin_weights"].view(B, n_bins), views["ori_vec"].view(B, 2)
    cabi.pose_labels(poses.to(dev), sigma, n_bins, gt, views["pyramid"], w, v)
    torch.cuda.synchronize()
    for k, buf in bufs.items():
        assert bool((buf[:guard] == sentinel).all()) and bool((buf[guard + sizes[k]:] == sentinel).all()), k
    return gt, views["pyramid"], w, v


def _gt_cases():
    cases = []
    for sigma in (1.0, 4.0, 40.0):
        p8 = synthetic_poses(8, seed=int(sigma))
        p8[0, :2] = torch.tensor([255.0, 256.0], dtype=torch.float64)        # integer centre
        p8[1, :2] = torch.tensor([0.0, 511.0], dtype=torch.float64)          # corner
        p8[2, :2] = torch.tensor([300.5, 12.75], dtype=torch.float64)        # fractional
        cases.append(("b8_512", p8, 512, 512, sigma))
        special = torch.tensor([(r, c, 90.0) for r, c in _SPECIAL_128x192], dtype=torch.float64)
        cases.append(("special_128x192", special, 128, 192, sigma))
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("name,poses,H,W,sigma", _gt_cases(), ids=lambda v: v if isinstance(v, str) else None)
def test_gt_and_pyramid_from_poses(cuda_device, name, poses, H, W, sigma):
    """gt equals NumPy float64 rounded once to float32 (NaN where NumPy gives NaN), the pyramid of the same launch equals
    gt_pyramid(gt) and F.max_pool2d, and nothing outside the four outputs is written."""
    B = poses.shape[0]
    gt, pyramid, _, _ = _labels_into_guarded(poses, H, W, sigma, 20, cuda_device)
    want = _np_gt(poses.tolist(), H, W, sigma)
    _assert_same_floats(gt, want, "gt", poses.tolist(), sigma)
    print("%s sigma=%g: %d gt elements compared, %d non-zero, %d NaN" % (
        name, sigma, want.numel(), int((want != 0).sum()), int(torch.isnan(want).sum())))
    if name.startswith("special"):
        assert bool(torch.isnan(want).any()) and bool((want == 0).any()) and bool((want == 1).any())
    ref = torch.empty_like(pyramid)
    cabi.gt_pyramid(gt, ref)
    _assert_same_floats(pyramid, ref, "pyramid vs gt_pyramid")
    off = 0
    for k in KS:
        n = B * (H // k) * (W // k)
        _assert_same_floats(pyramid[off:off + n].view(B, 1, H // k, W // k), F.max_pool2d(gt, k, stride=k), "k=%d" % k)
        off += n
    gt2, w2, v2, levels = losses.labels_from_poses(poses.to(cuda_device), (H, W), sigma)
    _assert_same_floats(gt2, want, "labels_from_poses gt")
    for got, k in zip(levels, KS):
        _assert_same_floats(got, F.max_pool2d(gt, k, stride=k), "labels_from_poses k=%d" % k)


# ---------------------------------------------------------------------------------------------------------------
# GPU: orientation labels
# ---------------------------------------------------------------------------------------------------------------
def _valid_angles():
    special = [0.0, -0.0, math.nextafter(360.0, 0.0)]
    for k in range(20):
        m = 18.0 * k
        special += [m, math.nextafter(m, 360.0)] + ([math.nextafter(m, -1.0)] if k else [])
    g = np.random.default_rng(5)
    near = (g.integers(0, 20, 20_000) * 18.0) + g.choice([-1.0, 1.0], 20_000) * 10.0 ** g.uniform(-15, -3, 20_000)
    near = near[(near >= 0) & (near < 360)]
    return special + near.tolist() + (g.random(85_000) * 360.0).tolist()


INVALID_ANGLES = [-1e-9, 360.0, INF, NAN, -INF, -5e-324, math.nextafter(360.0, 1e9), -18.0, 1e300, 720.0]


@pytest.mark.gpu
@pytest.mark.parametrize("n_bins", [10, 16, 20, 21, 32])
def test_orientation_labels_from_poses_are_bit_identical(cuda_device, n_bins):
    """Over 100 000 angles, including 0, -0.0, every multiple of 18 and its neighbours on both sides and the largest angle
    below 360: the weights and vectors are orientation_labels' bit for bit (signed zeros included); out-of-range and
    non-finite angles give NaN rows."""
    valid = _valid_angles()
    assert len(valid) >= 100_000
    angles = valid + INVALID_ANGLES
    want_w, want_v = losses.orientation_labels(valid, n_bins)
    got_w, got_v = [], []
    chunk = 40_000                                           # pairs per launch (at most 65535)
    for s in range(0, len(angles), chunk):
        a = torch.tensor(angles[s:s + chunk], dtype=torch.float64)
        poses = torch.stack([torch.full_like(a, 20.0), torch.full_like(a, 30.0), a], dim=1).to(cuda_device)
        _, w, v, _ = losses.labels_from_poses(poses, (64, 64), 4.0, n_bins)
        got_w.append(w.cpu())
        got_v.append(v.cpu())
    got_w, got_v = torch.cat(got_w), torch.cat(got_v)
    n = len(valid)
    for got, want, what in ((got_w[:n], want_w, "bin_weights"), (got_v[:n], want_v, "ori_vec")):
        bad = (got.view(torch.int32) != want.view(torch.int32)).any(dim=1)
        assert not bool(bad.any()), "%s differ for %d angles, e.g. %r" % (
            what, int(bad.sum()), [valid[i] for i in bad.nonzero().flatten()[:5].tolist()])
    assert bool(torch.isnan(got_w[n:]).all()) and bool(torch.isnan(got_v[n:]).all())
    print("n_bins=%d: %d angles compared bit for bit, %d NaN rows" % (n_bins, n, len(INVALID_ANGLES)))


# ---------------------------------------------------------------------------------------------------------------
# GPU: loss and gradients, graph replay
# ---------------------------------------------------------------------------------------------------------------
def _host_labels(poses, n_bins, size=512, sigma=4.0):
    gt = _np_gt(poses.tolist(), size, size, sigma)
    bin_weights, ori_vec = losses.orientation_labels(poses[:, 2], n_bins)
    return gt, bin_weights, ori_vec


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_training_loss_from_poses_equals_labels(cuda_device, precision):
    """CVM_VIGOR training outputs: training_loss_from_poses against training_loss_from_labels fed host-built labels
    (NumPy gt + orientation_labels).  Same loss, same gradient w.r.t. the eight outputs the loss reads, and the same
    gradient of every trainable parameter.  The encoders are frozen: the gradient they receive is the same either way, and
    PyTorch's cuDNN weight gradients are not bit-reproducible from one backward pass to the next."""
    dev = cuda_device
    B = 2
    model = build_model("vigor", None, True, 41).to(dev).set_precision(precision).eval()
    for n_, p_ in model.named_parameters():
        p_.requires_grad_("efficientnet" not in n_)
    params = [p_ for p_ in model.parameters() if p_.requires_grad]
    grd, sat = (t.to(dev) for t in synthetic_pair(B, GROUND_SHAPES["vigor"], seed=71))
    poses = synthetic_poses(B, seed=13)
    poses[1, :2] += torch.tensor([0.3, -0.45], dtype=torch.float64)   # centres off the float32 grid
    gt, bin_weights, ori_vec = (t.to(dev) for t in _host_labels(poses, 20))
    results = []
    for from_poses in (False, True):
        out = model(grd, sat)                                  # one forward per backward pass
        if from_poses:
            loss = losses.training_loss_from_poses(out, poses.to(dev))
        else:
            loss = losses.training_loss_from_labels(out, gt, bin_weights, ori_vec)
        wrt = [out[0], out[2]] + list(out[3:9])
        results.append((loss.detach(), torch.autograd.grad(loss, wrt + params)))
    (l_ref, g_ref), (l_got, g_got) = results
    assert torch.isfinite(l_ref) and torch.equal(l_got, l_ref), (l_got.item(), l_ref.item())
    assert len(params) > 90
    for i, (a, b) in enumerate(zip(g_got, g_ref)):
        assert a.dtype == b.dtype and torch.equal(a, b), i


@pytest.mark.gpu
def test_graphed_step_from_poses_with_inputs_rewritten(cuda_device):
    """training.GraphedTrainStep over (grd_u8, sat_u8, mats, poses): the step rotates the aerial on the device
    (affine_u8) and trains from poses.  The matrices and poses are rewritten in place before every replay, and each replay
    equals an eager step of an identical model on the same inputs: the same loss and, at the end, the same parameters."""
    from ccvpe_b200.training import GraphedTrainStep
    dev = cuda_device
    B, S = 2, 640
    g = np.random.default_rng(31)
    grd = torch.from_numpy(g.integers(0, 256, (B, 3, 320, 640), dtype=np.uint8)).to(dev)
    sat = torch.from_numpy(g.integers(0, 256, (B, S, S, 3), dtype=np.uint8)).to(dev)

    def draw():
        mats = torch.tensor([models.rotate_matrix(float(a), (S, S)) for a in g.uniform(-180, 180, B)], dtype=torch.float64)
        poses = torch.tensor([[g.uniform(40, 470), g.uniform(40, 470), g.uniform(0, 360)] for _ in range(B)],
                             dtype=torch.float64)
        return mats.to(dev), poses.to(dev)

    def make_step():
        model = build_model("vigor", None, True, 34).to(dev).set_precision("bf16").eval()
        for n_, p_ in model.named_parameters():
            p_.requires_grad_("efficientnet" not in n_)
        opt = torch.optim.Adam([p_ for p_ in model.parameters() if p_.requires_grad], lr=1e-4, fused=True,
                               capturable=True)

        def fn(grd_u8, sat_u8, mats, poses):
            opt.zero_grad(set_to_none=False)
            sat_rot = model.affine_u8(sat_u8, mats, (512, 512), offset=(64, 64))
            loss = losses.training_loss_from_poses(model(grd_u8, sat_rot), poses)
            loss.backward()
            opt.step()
            return loss.detach()
        return model, fn

    first = [grd, sat, *draw()]
    model_e, eager = make_step()
    model_g, fn_g = make_step()
    for _ in range(2):
        eager(*first)                                          # the graph side's step 1 and warm-up step
    fn_g(*first)
    step = GraphedTrainStep(fn_g, first, warmup=1)
    mats_s, poses_s = step.static_in[2], step.static_in[3]
    for i in range(4):
        mats, poses = draw()
        mats_s.copy_(mats)                                     # in place: the replay reads them when it runs
        poses_s.copy_(poses)
        got = step(*step.static_in).clone()
        want = eager(grd, sat, mats, poses)
        torch.cuda.synchronize()
        assert torch.isfinite(want) and torch.equal(got, want), (i, got.item(), want.item())
    for (n_, a), b in zip(model_g.named_parameters(), model_e.parameters()):
        assert torch.equal(a, b), n_
