"""Drop-in replacements of the reference's training losses (reference losses.py:4-29), each ONE fused CUDA call that
produces the loss value and its gradient (libccvpe_b200: ccvpe_infonce_loss / ccvpe_cross_entropy_loss /
ccvpe_orientation_loss).  Same names, argument order and semantics as the reference, so train_VIGOR.py:137-146 reads

    loss_ori = orientation_loss(ori, gt_orientation, gt)
    loss_infoNCE = infoNCELoss(torch.flatten(matching_score_stacked, start_dim=1), torch.flatten(gt_bottleneck, start_dim=1))
    loss_ce = cross_entropy_loss(logits_flattened, gt_flattened)

unchanged.  Labels / ground-truth maps are treated as constants (they are data in the reference too); there is no CPU path.
"""
from __future__ import annotations

import math

import torch

from . import cabi


def _f32c(t: torch.Tensor) -> torch.Tensor:
    return t.detach().contiguous().float()


class _InfoNCE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, scores, labels, temperature):
        if not scores.is_cuda:
            raise cabi.CcvpeError("ccvpe_b200.losses run on CUDA only; there is no CPU fallback")
        s, l = _f32c(scores), _f32c(labels)
        loss = torch.empty((), dtype=torch.float32, device=s.device)
        ds = torch.empty_like(s)
        with cabi.device_of(s):
            cabi.infonce_loss(s, l, float(temperature), loss, ds)
        ctx.save_for_backward(ds)
        return loss

    @staticmethod
    def backward(ctx, g):
        (ds,) = ctx.saved_tensors
        return ds * g, None, None


class _CrossEntropy(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, labels):
        if not logits.is_cuda:
            raise cabi.CcvpeError("ccvpe_b200.losses run on CUDA only; there is no CPU fallback")
        x, l = _f32c(logits), _f32c(labels)
        loss = torch.empty((), dtype=torch.float32, device=x.device)
        dx = torch.empty_like(x)
        with cabi.device_of(x):
            cabi.cross_entropy_loss(x, l, loss, dx)
        ctx.save_for_backward(dx)
        return loss

    @staticmethod
    def backward(ctx, g):
        (dx,) = ctx.saved_tensors
        return dx * g, None


class _Orientation(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ori, gt_orientation, gt):
        if not ori.is_cuda:
            raise cabi.CcvpeError("ccvpe_b200.losses run on CUDA only; there is no CPU fallback")
        o, go, w = _f32c(ori), _f32c(gt_orientation), _f32c(gt)
        loss = torch.empty((), dtype=torch.float32, device=o.device)
        do = torch.empty_like(o)
        with cabi.device_of(o):
            cabi.orientation_loss(o, go, w, loss, do)
        ctx.save_for_backward(do)
        return loss

    @staticmethod
    def backward(ctx, g):
        (do,) = ctx.saved_tensors
        return do * g, None, None


class _InfoNCEBinned(torch.autograd.Function):
    @staticmethod
    def forward(ctx, scores, gt_pooled, bin_weights, temperature):
        if not scores.is_cuda:
            raise cabi.CcvpeError("ccvpe_b200.losses run on CUDA only; there is no CPU fallback")
        s = _f32c(scores)
        loss = torch.empty((), dtype=torch.float32, device=s.device)
        ds = torch.empty_like(s)
        with cabi.device_of(s):
            cabi.infonce_loss_binned(s, _f32c(gt_pooled), _f32c(bin_weights), float(temperature), loss, ds)
        ctx.save_for_backward(ds)
        return loss

    @staticmethod
    def backward(ctx, g):
        (ds,) = ctx.saved_tensors
        return ds * g, None, None, None


class _OrientationConst(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ori, ori_vec, gt):
        if not ori.is_cuda:
            raise cabi.CcvpeError("ccvpe_b200.losses run on CUDA only; there is no CPU fallback")
        o = _f32c(ori)
        loss = torch.empty((), dtype=torch.float32, device=o.device)
        do = torch.empty_like(o)
        with cabi.device_of(o):
            cabi.orientation_loss_const(o, _f32c(ori_vec), _f32c(gt), loss, do)
        ctx.save_for_backward(do)
        return loss

    @staticmethod
    def backward(ctx, g):
        (do,) = ctx.saved_tensors
        return do * g, None, None


def infoNCELoss(scores, labels, temperature=0.1):
    """reference losses.py:4-20 -- weighted InfoNCE over a flattened score volume [B, n]; positives = labels > 1e-2."""
    return _InfoNCE.apply(scores, labels, temperature)


def cross_entropy_loss(logits, labels):
    """reference losses.py:23-24 -- -sum(labels * log_softmax(logits, dim=1)) / B."""
    return _CrossEntropy.apply(logits, labels)


def orientation_loss(ori, gt_orientation, gt):
    """reference losses.py:28-29 -- sum(sum((gt_orientation - ori)^2, dim=1, keepdim=True) * gt) / B;
    ori, gt_orientation [B, 2, H, W], gt [B, 1, H, W]."""
    return _Orientation.apply(ori, gt_orientation, gt)


def training_loss(outputs, gt, gt_with_ori, gt_orientation, weight_infoNCE=1e4, weight_ori=1e1):
    """The reference's loss combination (train_VIGOR.py:120-146) on the 9-tuple a model returns: GT preparation
    (flatten + normalise `gt`; max-pool `gt_with_ori` to the six score-volume resolutions) and
    loss_ce + weight_infoNCE * mean(infoNCE_1..6) + weight_ori * loss_ori."""
    logits_flattened, _heatmap, ori = outputs[0], outputs[1], outputs[2]
    gt_flattened = torch.flatten(gt, start_dim=1)
    gt_flattened = gt_flattened / torch.sum(gt_flattened, dim=1, keepdim=True)
    loss_ori = orientation_loss(ori, gt_orientation, gt)
    nce = 0
    for scores, k in zip(outputs[3:9], (64, 32, 16, 8, 4, 2)):
        gt_b = torch.nn.functional.max_pool2d(gt_with_ori, k, stride=k)
        nce = nce + infoNCELoss(torch.flatten(scores, start_dim=1), torch.flatten(gt_b, start_dim=1))
    loss_ce = cross_entropy_loss(logits_flattened, gt_flattened)
    return loss_ce + weight_infoNCE * nce / 6 + weight_ori * loss_ori


# ------------------------------------------------------------------------------------------------------------------
# Compact labels.  A pair's orientation-binned map is rank 1 and its orientation field is constant:
#     gt_with_ori    = gt * bin_weights[:, :, None, None]              gt [B, 1, H, W], bin_weights [B, R]
#     gt_orientation = ori_vec[:, :, None, None].expand(B, 2, H, W)    ori_vec [B, 2]
# so a training batch can carry (gt, bin_weights, ori_vec) instead of the 23 MiB of maps per 512x512 pair.  The losses below
# read the factors directly and give the same loss and gradient bits as `training_loss` on the materialised maps.
# ------------------------------------------------------------------------------------------------------------------
def orientation_labels(angles_deg, n_bins=20):
    """VIGOR's 18-degree orientation rule (reference datasets.py:142-166, as `synthetic.synthetic_ground_truth` writes it)
    for a batch of angles in degrees (a sequence of floats or a CPU tensor): returns CPU fp32 tensors
    bin_weights [B, n_bins] and ori_vec [B, 2].

    index = int(angle // 18) and ratio = (angle % 18) / 18 split the pair over two adjacent bins with weights 1 - ratio and
    ratio: bins 0 and n_bins - 1 when index == 0, otherwise n_bins - index and n_bins - index - 1 (negative bins count
    from the end, as tensor indexing does); ori_vec = (cos, sin) of the angle.  Computed in Python float arithmetic, as the
    dense maps are.  Datasets with another rule pass their own non-negative per-pair weights instead."""
    angles = angles_deg.tolist() if isinstance(angles_deg, torch.Tensor) else [float(a) for a in angles_deg]
    bin_weights = torch.zeros(len(angles), n_bins)
    ori_vec = torch.zeros(len(angles), 2)
    for b, angle in enumerate(angles):
        index, ratio = int(angle // 18), (angle % 18) / 18
        lo, hi = (0, n_bins - 1) if index == 0 else (n_bins - index, n_bins - index - 1)
        bin_weights[b, lo] = 1 - ratio
        bin_weights[b, hi] = ratio
        ori_vec[b, 0] = math.cos(math.radians(angle))
        ori_vec[b, 1] = math.sin(math.radians(angle))
    return bin_weights, ori_vec


def gt_pyramid(gt):
    """The six InfoNCE label maps of `gt` [B, 1, H, W] (H, W multiples of 64): [max_pool2d(gt, k, stride=k) for k in
    (64, 32, 16, 8, 4, 2)], computed by one kernel launch.  Views into one buffer."""
    if not gt.is_cuda:
        raise cabi.CcvpeError("ccvpe_b200.losses run on CUDA only; there is no CPU fallback")
    g = _f32c(gt)
    B, _, H, W = g.shape
    out = torch.empty(cabi.gt_pyramid_elems(B, H, W), dtype=torch.float32, device=g.device)
    with cabi.device_of(g):
        cabi.gt_pyramid(g, out)
    levels, off = [], 0
    for k in cabi.GT_PYRAMID_KS:
        n = B * (H // k) * (W // k)
        levels.append(out[off:off + n].view(B, 1, H // k, W // k))
        off += n
    return levels


def infoNCELoss_binned(scores, gt_pooled, bin_weights, temperature=0.1):
    """infoNCELoss(flatten(scores), flatten(gt_pooled * bin_weights[:, :, None, None])) without materialising the labels:
    scores [B, R, h, w], gt_pooled [B, 1, h, w], bin_weights [B, R]."""
    return _InfoNCEBinned.apply(scores, gt_pooled, bin_weights, temperature)


def orientation_loss_const(ori, ori_vec, gt):
    """orientation_loss(ori, ori_vec[:, :, None, None].expand_as(ori), gt): ori [B, 2, H, W], ori_vec [B, 2],
    gt [B, 1, H, W]."""
    return _OrientationConst.apply(ori, ori_vec, gt)


def training_loss_from_labels(outputs, gt, bin_weights, ori_vec, weight_infoNCE=1e4, weight_ori=1e1):
    """`training_loss` on compact labels: gt [B, 1, H, W], bin_weights [B, R], ori_vec [B, 2] (device tensors; see
    `orientation_labels`).  Same value and gradients as training_loss(outputs, gt, gt * bin_weights[:, :, None, None],
    ori_vec[:, :, None, None].expand(B, 2, H, W)); one label-pyramid launch replaces the six max-pools.  Every score volume
    must have bin_weights.shape[1] orientation channels."""
    logits_flattened, _heatmap, ori = outputs[0], outputs[1], outputs[2]
    for level, scores in enumerate(outputs[3:9], start=1):
        if scores.dim() != 4 or scores.shape[1] != bin_weights.shape[1]:
            raise cabi.CcvpeError("training_loss_from_labels: score volume %d has shape %s, but bin_weights has %d bins "
                                  "(each level needs one weight per orientation channel)"
                                  % (level, tuple(scores.shape), bin_weights.shape[1]))
    gt_flattened = torch.flatten(gt, start_dim=1)
    gt_flattened = gt_flattened / torch.sum(gt_flattened, dim=1, keepdim=True)
    loss_ori = orientation_loss_const(ori, ori_vec, gt)
    nce = 0
    for scores, gt_b in zip(outputs[3:9], gt_pyramid(gt)):
        nce = nce + infoNCELoss_binned(scores, gt_b, bin_weights)
    loss_ce = cross_entropy_loss(logits_flattened, gt_flattened)
    return loss_ce + weight_infoNCE * nce / 6 + weight_ori * loss_ori
