"""Training from compact labels: (gt, bin_weights, ori_vec) instead of the dense gt_with_ori / gt_orientation maps.

CPU: the label helper and the synthetic data reproduce the dense maps bit for bit (against verbatim copies of the previous
dense implementation), and the bindings refuse bad arguments before launching.  GPU: the label pyramid equals
F.max_pool2d, and the compact-label losses give the same loss and gradient bits (torch.equal) as the dense-label losses
fed the materialised maps."""
import ctypes
import math

import pytest
import torch
from torch.nn import functional as F

from ccvpe_b200 import cabi, losses
from ccvpe_b200.synthetic import GROUND_SHAPES, synthetic_ground_truth, synthetic_labels, synthetic_pair
from helpers import build_model

KS = (64, 32, 16, 8, 4, 2)


# ---------------------------------------------------------------------------------------------------------------
# verbatim copies of the dense ground truth as it was built before compact labels existed
# ---------------------------------------------------------------------------------------------------------------
def _dense_ground_truth_before(batch: int, seed: int = 0, size: int = 512, n_bins: int = 20):
    g = torch.Generator().manual_seed(20_000 + seed)
    ys = torch.arange(size, dtype=torch.float32).view(size, 1)
    xs = torch.arange(size, dtype=torch.float32).view(1, size)
    gt = torch.zeros(batch, 1, size, size)
    gt_with_ori = torch.zeros(batch, n_bins, size, size)
    gt_orientation = torch.zeros(batch, 2, size, size)
    for b in range(batch):
        cy, cx = (torch.rand(2, generator=g) * (size - 64) + 32).tolist()
        blob = torch.exp(-((ys - cy) ** 2 + (xs - cx) ** 2) / (2.0 * 4.0 ** 2))
        gt[b, 0] = blob
        angle = float(torch.rand(1, generator=g)) * 360.0
        index, ratio = int(angle // 18), (angle % 18) / 18
        if index == 0:
            gt_with_ori[b, 0] = blob * (1 - ratio)
            gt_with_ori[b, n_bins - 1] = blob * ratio
        else:
            gt_with_ori[b, n_bins - index] = blob * (1 - ratio)
            gt_with_ori[b, n_bins - index - 1] = blob * ratio
        gt_orientation[b, 0] = math.cos(math.radians(angle))
        gt_orientation[b, 1] = math.sin(math.radians(angle))
    return gt, gt_with_ori, gt_orientation


def _dense_pair_before(blob, angle, gt_with_ori, gt_orientation, b, n_bins):
    """The per-pair loop body above, verbatim, for a given blob and angle."""
    index, ratio = int(angle // 18), (angle % 18) / 18
    if index == 0:
        gt_with_ori[b, 0] = blob * (1 - ratio)
        gt_with_ori[b, n_bins - 1] = blob * ratio
    else:
        gt_with_ori[b, n_bins - index] = blob * (1 - ratio)
        gt_with_ori[b, n_bins - index - 1] = blob * ratio
    gt_orientation[b, 0] = math.cos(math.radians(angle))
    gt_orientation[b, 1] = math.sin(math.radians(angle))


def _expand(gt, bin_weights, ori_vec):
    B, _, H, W = gt.shape
    return gt * bin_weights[:, :, None, None], ori_vec[:, :, None, None].expand(B, 2, H, W)


# ---------------------------------------------------------------------------------------------------------------
# CPU: label helper and synthetic data
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("batch,seed,size,n_bins", [(3, 0, 512, 20), (4, 7, 128, 16), (2, 11, 64, 20)])
def test_synthetic_ground_truth_unchanged(batch, seed, size, n_bins):
    got = synthetic_ground_truth(batch, seed=seed, size=size, n_bins=n_bins)
    want = _dense_ground_truth_before(batch, seed=seed, size=size, n_bins=n_bins)
    for a, b in zip(got, want):
        assert a.dtype == b.dtype and a.shape == b.shape and torch.equal(a, b)


@pytest.mark.parametrize("batch,seed,n_bins", [(3, 0, 20), (5, 3, 16)])
def test_synthetic_labels_expand_to_the_dense_maps(batch, seed, n_bins):
    gt, angles = synthetic_labels(batch, seed=seed, size=128)
    assert angles.dtype == torch.float64 and angles.shape == (batch,)
    bin_weights, ori_vec = losses.orientation_labels(angles, n_bins)
    assert bin_weights.shape == (batch, n_bins) and ori_vec.shape == (batch, 2)
    assert bin_weights.dtype == ori_vec.dtype == torch.float32 and not bin_weights.is_cuda
    d_gt, d_gwo, d_gor = synthetic_ground_truth(batch, seed=seed, size=128, n_bins=n_bins)
    gwo, gor = _expand(gt, bin_weights, ori_vec)
    assert torch.equal(gt, d_gt) and torch.equal(gwo, d_gwo) and torch.equal(gor, d_gor)


@pytest.mark.parametrize("n_bins", [20, 16])
def test_orientation_labels_at_bin_edges(n_bins):
    angles = [0.0, 1e-6, 17.999999, 18.0, 179.5, 342.0, 359.999999]
    ys = torch.arange(64, dtype=torch.float32).view(64, 1)
    xs = torch.arange(64, dtype=torch.float32).view(1, 64)
    blob = torch.exp(-((ys - 30.3) ** 2 + (xs - 21.7) ** 2) / (2.0 * 4.0 ** 2))
    B = len(angles)
    want_gwo = torch.zeros(B, n_bins, 64, 64)
    want_gor = torch.zeros(B, 2, 64, 64)
    for b, angle in enumerate(angles):
        _dense_pair_before(blob, angle, want_gwo, want_gor, b, n_bins)
    for given in (angles, torch.tensor(angles, dtype=torch.float64)):
        bin_weights, ori_vec = losses.orientation_labels(given, n_bins)
        assert int((bin_weights != 0).sum(dim=1).max()) <= 2
        gwo, gor = _expand(blob.expand(B, 1, 64, 64), bin_weights, ori_vec)
        assert torch.equal(gwo, want_gwo) and torch.equal(gor, want_gor)


# ---------------------------------------------------------------------------------------------------------------
# CPU: argument checks before any launch
# ---------------------------------------------------------------------------------------------------------------
def _cpu_loss_args(B=2, R=20, h=8, w=8):
    return dict(scores=torch.zeros(B, R, h, w), pooled=torch.zeros(B, 1, h, w), bin_w=torch.zeros(B, R),
                temperature=0.1, loss=torch.zeros(()), d_scores=torch.zeros(B, R, h, w))


def test_gt_pyramid_binding_refuses_bad_arguments():
    gt = torch.zeros(2, 1, 128, 192)
    out = torch.zeros(cabi.gt_pyramid_elems(2, 128, 192))
    cases = [
        (gt.double(), out, "float32"),
        (gt[:, 0], out, "shape"),
        (torch.zeros(2, 1, 192, 128).transpose(2, 3), out, "contiguous"),
        (torch.zeros(2, 1, 96, 192), torch.zeros(cabi.gt_pyramid_elems(2, 96, 192)), "multiples of 64"),
        (torch.zeros(2, 1, 128, 200), torch.zeros(cabi.gt_pyramid_elems(2, 128, 200)), "multiples of 64"),
        (gt, out[1:], "shape"),
        (gt, out.half(), "float32"),
        (gt, out, "CUDA"),                       # well-formed CPU tensors: refused for the device, never launched
    ]
    for g, o, msg in cases:
        with pytest.raises(cabi.CcvpeError, match=msg):
            cabi.gt_pyramid(g, o)


def test_binned_loss_bindings_refuse_bad_arguments():
    def call(**kw):
        a = _cpu_loss_args()
        a.update(kw)
        cabi.infonce_loss_binned(a["scores"], a["pooled"], a["bin_w"], a["temperature"], a["loss"], a["d_scores"])

    with pytest.raises(cabi.CcvpeError, match="scores must be a float32"):
        call(scores=torch.zeros(2, 20, 8, 8, dtype=torch.bfloat16))
    with pytest.raises(cabi.CcvpeError, match="gt_pooled must have shape"):
        call(pooled=torch.zeros(2, 1, 8, 16))
    with pytest.raises(cabi.CcvpeError, match="bin_weights must have shape"):
        call(bin_w=torch.zeros(2, 16))
    with pytest.raises(cabi.CcvpeError, match="contiguous"):
        call(scores=torch.zeros(2, 20, 8, 8).transpose(2, 3))
    with pytest.raises(cabi.CcvpeError, match="d_scores must have shape"):
        call(d_scores=torch.zeros(2, 20, 64))
    with pytest.raises(cabi.CcvpeError, match="CUDA"):
        call()

    def call_ori(**kw):
        a = dict(ori=torch.zeros(2, 2, 64, 64), ori_vec=torch.zeros(2, 2), gt=torch.zeros(2, 1, 64, 64),
                 loss=torch.zeros(()), d_ori=torch.zeros(2, 2, 64, 64))
        a.update(kw)
        cabi.orientation_loss_const(a["ori"], a["ori_vec"], a["gt"], a["loss"], a["d_ori"])

    with pytest.raises(cabi.CcvpeError, match="ori_vec must have shape"):
        call_ori(ori_vec=torch.zeros(2, 2, 1, 1))
    with pytest.raises(cabi.CcvpeError, match="gt must have shape"):
        call_ori(gt=torch.zeros(2, 1, 64, 32))
    with pytest.raises(cabi.CcvpeError, match="ori_vec must be a float32"):
        call_ori(ori_vec=torch.zeros(2, 2, dtype=torch.float64))
    with pytest.raises(cabi.CcvpeError, match="contiguous"):
        call_ori(ori=torch.zeros(2, 64, 64, 2).permute(0, 3, 1, 2))
    with pytest.raises(cabi.CcvpeError, match="CUDA"):
        call_ori()


def test_c_abi_refuses_bad_sizes_before_launch():
    """The C entry points check their sizes before touching memory or the device (the pointers are never dereferenced)."""
    lib = cabi.load()
    p = ctypes.c_void_p(4096)
    bad = -1                                                                    # CCVPE_ERR_BAD_ARGUMENT
    for B, H, W in [(1, 100, 128), (1, 128, 96), (2, 0, 64), (0, 64, 64), (1, -64, 64)]:
        assert lib.ccvpe_gt_pyramid(p, B, H, W, p, None) == bad, (B, H, W)
        assert b"multiples of 64" in lib.ccvpe_last_error()
    assert lib.ccvpe_gt_pyramid(ctypes.c_void_p(4100), 1, 64, 64, p, None) == bad        # gt not 16-byte aligned
    assert lib.ccvpe_infonce_loss_binned(p, p, p, 1, 20, 1 << 27, ctypes.c_float(0.1), p, p, p, None) == bad
    assert lib.ccvpe_infonce_loss_binned(p, p, p, 1, 0, 64, ctypes.c_float(0.1), p, p, p, None) == bad
    assert lib.ccvpe_orientation_loss_const(p, None, p, 1, 64, p, p, p, None) == bad


def test_training_loss_from_labels_refuses_mismatched_bins():
    """CVM_VIGOR_ori_prior's levels carry 2k+1 orientation channels, not one per bin: refused, naming the level."""
    B = 1
    outputs = [torch.zeros(B, 512 * 512), torch.zeros(B, 1, 512, 512), torch.zeros(B, 2, 512, 512)]
    outputs += [torch.zeros(B, 9 if level == 3 else 20, 512 // k, 512 // k) for level, k in enumerate(KS, start=1)]
    gt = torch.zeros(B, 1, 512, 512)
    with pytest.raises(cabi.CcvpeError, match="score volume 3 has shape"):
        losses.training_loss_from_labels(outputs, gt, torch.zeros(B, 20), torch.zeros(B, 2))
    with pytest.raises(cabi.CcvpeError, match="score volume 1 has shape"):
        losses.training_loss_from_labels(outputs, gt, torch.zeros(B, 16), torch.zeros(B, 2))


# ---------------------------------------------------------------------------------------------------------------
# GPU: label pyramid
# ---------------------------------------------------------------------------------------------------------------
def _pyramid_input(kind, B, H, W, g):
    if kind == "blobs":
        ys = torch.arange(H, dtype=torch.float32).view(H, 1)
        xs = torch.arange(W, dtype=torch.float32).view(1, W)
        gt = torch.zeros(B, 1, H, W)
        for b in range(B):
            for _ in range(3):
                cy, cx = (torch.rand(2, generator=g) * torch.tensor([H, W])).tolist()
                gt[b, 0] += torch.exp(-((ys - cy) ** 2 + (xs - cx) ** 2) / (2.0 * 4.0 ** 2))
        return gt
    gt = torch.rand(B, 1, H, W, generator=g) * 2 - 1
    if kind == "special":
        flat = gt.view(-1)
        n = flat.numel()
        flat[torch.randint(0, n, (max(1, n // 3000),), generator=g)] = float("inf")
        flat[torch.randint(0, n, (max(1, n // 3000),), generator=g)] = float("-inf")
        flat[torch.randint(0, n, (max(1, n // 2000),), generator=g)] = float("nan")
    return gt


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["blobs", "noise", "special"])
@pytest.mark.parametrize("H,W", [(512, 512), (128, 192)])
@pytest.mark.parametrize("B", [1, 3, 8])
def test_gt_pyramid_equals_max_pool2d(cuda_device, B, H, W, kind):
    dev = cuda_device
    g = torch.Generator().manual_seed(1000 * B + H + W + len(kind))
    gt = _pyramid_input(kind, B, H, W, g).to(dev)
    n, guard = cabi.gt_pyramid_elems(B, H, W), 4096
    sentinel = -1234.5
    buf = torch.full((n + 2 * guard,), sentinel, device=dev)
    cabi.gt_pyramid(gt, buf[guard:guard + n])
    torch.cuda.synchronize()
    assert bool((buf[:guard] == sentinel).all()) and bool((buf[guard + n:] == sentinel).all())
    off = 0
    for k in KS:
        m = B * (H // k) * (W // k)
        got = buf[guard + off:guard + off + m].view(B, 1, H // k, W // k)
        want = F.max_pool2d(gt, k, stride=k)
        nan = torch.isnan(want)
        assert torch.equal(torch.isnan(got), nan), k
        assert torch.equal(got[~nan], want[~nan]), k
        if kind == "special" and k == 64:
            assert bool(nan.any())                   # the planted NaNs do reach the coarsest level
        off += m
    assert off == n
    for got, k in zip(losses.gt_pyramid(gt), KS):   # the public wrapper's views
        want = F.max_pool2d(gt, k, stride=k)
        nan = torch.isnan(want)
        assert got.shape == want.shape and torch.equal(torch.isnan(got), nan) and torch.equal(got[~nan], want[~nan])


# ---------------------------------------------------------------------------------------------------------------
# GPU: losses on compact labels vs dense labels
# ---------------------------------------------------------------------------------------------------------------
def _bin_weights(B, R, g):
    """Per-pair two-bin weights from random angles; pair 0 sits exactly on a bin edge, so one of its weights is zero."""
    angles = (torch.rand(B, generator=g, dtype=torch.float64) * 360.0).tolist()
    angles[0] = 36.0
    w, _ = losses.orientation_labels(angles, R)
    assert int((w[0] != 0).sum()) == 1
    return w


@pytest.mark.gpu
@pytest.mark.parametrize("R", [20, 16])
@pytest.mark.parametrize("B", [1, 8])
@pytest.mark.parametrize("hw", [8, 16, 32, 64, 128, 256])
def test_infonce_binned_equals_dense(cuda_device, B, R, hw):
    dev = cuda_device
    g = torch.Generator().manual_seed(17 * B + R + hw)
    scores = (torch.rand(B, R, hw, hw, generator=g) * 2 - 1).to(dev)
    # pooled labels around the 1e-2 / w positive threshold: some products land on either side of it
    pooled = (torch.rand(B, 1, hw, hw, generator=g) * 0.04).to(dev)
    w = _bin_weights(B, R, g).to(dev)
    labels = pooled * w[:, :, None, None]
    assert bool((labels > 1e-2).any()) and bool(((labels > 0) & (labels <= 1e-2)).any())
    sd = scores.clone().requires_grad_(True)
    ref = losses.infoNCELoss(torch.flatten(sd, start_dim=1), torch.flatten(labels, start_dim=1))
    (d_ref,) = torch.autograd.grad(ref, sd)
    sb = scores.clone().requires_grad_(True)
    got = losses.infoNCELoss_binned(sb, pooled, w)
    (d_got,) = torch.autograd.grad(got, sb)
    assert torch.equal(got, ref), (got.item(), ref.item())
    assert torch.equal(d_got, d_ref)


@pytest.mark.gpu
@pytest.mark.parametrize("B,size", [(1, 512), (3, 512), (2, 128)])
def test_orientation_loss_const_equals_dense(cuda_device, B, size):
    dev = cuda_device
    g = torch.Generator().manual_seed(B * size)
    gt, angles = synthetic_labels(B, seed=B, size=size)
    _, ori_vec = losses.orientation_labels(angles)
    ori = F.normalize(torch.randn(B, 2, size, size, generator=g), dim=1).to(dev)
    gt, ori_vec = gt.to(dev), ori_vec.to(dev)
    od = ori.clone().requires_grad_(True)
    ref = losses.orientation_loss(od, ori_vec[:, :, None, None].expand(B, 2, size, size).contiguous(), gt)
    (d_ref,) = torch.autograd.grad(ref, od)
    oc = ori.clone().requires_grad_(True)
    got = losses.orientation_loss_const(oc, ori_vec, gt)
    (d_got,) = torch.autograd.grad(got, oc)
    assert torch.equal(got, ref) and torch.equal(d_got, d_ref)


@pytest.mark.gpu
@pytest.mark.parametrize("variant,shape_key,B,precision,n_bins", [
    ("vigor", "vigor", 2, "fp32", 20), ("vigor", "vigor", 2, "bf16", 20), ("kitti", "kitti", 1, "fp32", 16),
    ("oxford", "oxford", 1, "fp32", 20),
])
def test_training_loss_from_labels_equals_dense(cuda_device, variant, shape_key, B, precision, n_bins):
    """Value and autograd gradients w.r.t. the eight outputs the loss reads (logits, orientation field, six score volumes)
    of training_loss_from_labels vs training_loss on the equivalent dense maps, on real model outputs."""
    dev = cuda_device
    model = build_model(variant, None, True if variant == "vigor" else None, 41).to(dev).set_precision(precision)
    grd, sat = synthetic_pair(B, GROUND_SHAPES[shape_key], seed=71)
    with torch.no_grad():
        out = model(grd.to(dev), sat.to(dev))
    gt, angles = synthetic_labels(B, seed=13)
    bin_weights, ori_vec = losses.orientation_labels(angles, n_bins)
    gwo, gor = _expand(gt, bin_weights, ori_vec)
    gt, bin_weights, ori_vec, gwo, gor = (t.to(dev) for t in (gt, bin_weights, ori_vec, gwo, gor))
    assert all(s.shape[1] == n_bins for s in out[3:9])
    results = []
    for dense in (True, False):
        leaves = [t.detach().clone().requires_grad_(i != 1) for i, t in enumerate(out)]
        if dense:
            loss = losses.training_loss(leaves, gt, gwo, gor)
        else:
            loss = losses.training_loss_from_labels(leaves, gt, bin_weights, ori_vec)
        wrt = [leaves[0], leaves[2]] + leaves[3:9]
        results.append((loss.detach(), torch.autograd.grad(loss, wrt)))
    (l_d, g_d), (l_c, g_c) = results
    assert torch.isfinite(l_d) and torch.equal(l_c, l_d), (l_c.item(), l_d.item())
    for i, (a, b) in enumerate(zip(g_c, g_d)):
        assert a.dtype == b.dtype and torch.equal(a, b), i


@pytest.mark.gpu
def test_graphed_training_step_on_compact_labels_matches_eager(cuda_device):
    """training.GraphedTrainStep with (grd, sat, gt, bin_weights, ori_vec) as the step's inputs gives the same losses as
    the same steps run eagerly (same check and tolerance as the dense-label graph test)."""
    from ccvpe_b200.training import GraphedTrainStep
    dev = cuda_device
    gt, angles = synthetic_labels(2, seed=8)
    bin_weights, ori_vec = losses.orientation_labels(angles)
    batch = [t.to(dev) for t in synthetic_pair(2, (320, 640), seed=64)] + [t.to(dev) for t in (gt, bin_weights, ori_vec)]
    hist = {}
    for mode in ("eager", "graph"):
        model = build_model("vigor", None, True, 34).to(dev).set_precision("bf16").eval()
        for n_, p_ in model.named_parameters():
            p_.requires_grad_("._fc." not in n_)
        opt = torch.optim.Adam([p_ for p_ in model.parameters() if p_.requires_grad], lr=1e-4, fused=True, capturable=True)

        def fn(grd, sat, gt, w, v):
            opt.zero_grad(set_to_none=False)
            loss = losses.training_loss_from_labels(model(grd, sat), gt, w, v)
            loss.backward()
            opt.step()
            return loss.detach()

        if mode == "eager":
            hist[mode] = [float(fn(*batch)) for _ in range(6)]
        else:
            fn(*batch)                                               # step 1
            step = GraphedTrainStep(fn, batch, warmup=1)            # step 2 (warm-up); the capture itself executes nothing
            hist[mode] = [float("nan")] * 2 + [float(step(*batch)) for _ in range(4)]      # steps 3..6 are replays
    for a, b in zip(hist["eager"][2:], hist["graph"][2:]):
        assert abs(a - b) <= 1e-3 * abs(a), hist
    assert hist["eager"][-1] < hist["eager"][0]
