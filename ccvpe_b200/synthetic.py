"""Deterministic synthetic weights and inputs (there is no network for checkpoints or datasets).

`fill_deterministic` overwrites every tensor of a `state_dict` from a per-key seeded CPU generator, so two
models with the same state_dict keys (the reference's and ours) get bit-identical weights regardless of how
many random numbers their constructors consumed (SURVEY.md section 8(c) "Identical weights").  Scales are
He-style so activations keep O(1) magnitude through the 12-conv decoders and the 512x512 heatmap has a
well separated maximum (the reference's default init gives an almost flat heatmap, top-2 logit gap 8.6e-5,
which makes end-to-end argmax comparisons meaningless -- SURVEY.md section 7.3-4).
"""
from __future__ import annotations

import zlib
from typing import Dict

import torch

from .losses import orientation_labels

#: input shapes (H, W) of the ground image per dataset family; aerial is always 512x512
GROUND_SHAPES = {"vigor": (320, 640), "vigor_fov180": (320, 320), "vigor_fov108": (320, 192),
                 "kitti": (256, 1024), "oxford": (154, 231)}
AERIAL_SHAPE = (512, 512)


def _gen(seed: int, key: str) -> torch.Generator:
    g = torch.Generator(device="cpu")
    g.manual_seed((int(seed) * 1000003 + zlib.crc32(key.encode())) % (2 ** 63 - 1))
    return g


@torch.no_grad()
def fill_deterministic(state_dict: Dict[str, torch.Tensor], seed: int = 0) -> Dict[str, torch.Tensor]:
    """In-place, returns the same dict.  Works on a module's `state_dict()` (tensors alias the parameters)."""
    for key, t in state_dict.items():
        if not t.is_floating_point():
            continue
        g = _gen(seed, key)
        leaf = key.rsplit(".", 1)[-1]
        if leaf == "running_var":
            v = 1.0 + 0.1 * torch.rand(t.shape, generator=g)
        elif leaf == "running_mean":
            v = 0.1 * torch.randn(t.shape, generator=g)
        elif t.dim() == 1 and leaf == "weight":          # BatchNorm scale
            v = 1.0 + 0.1 * torch.randn(t.shape, generator=g)
        elif leaf == "bias":
            v = 0.05 * torch.randn(t.shape, generator=g)
        else:                                            # conv / deconv / linear weight
            if ".deconv" in "." + key or key.startswith("deconv"):
                fan_in = t.shape[0]                      # ConvTranspose2d weight is [Cin, Cout, 2, 2]; k2 s2 -> 1 tap/output
                gain = 1.0
            else:
                fan_in = t[0].numel()
                gain = 2.0
            if t.dim() == 4 and t.shape[0] <= 2 and t.shape[-1] == 3:
                gain *= 36.0                             # final 16->1 / 16->2 convs: plant a clearly peaked heatmap
            v = torch.randn(t.shape, generator=g) * (gain / max(fan_in, 1)) ** 0.5
        t.copy_(v.to(t.dtype))
    return state_dict


def synthetic_pair(batch: int, ground_hw, seed: int = 0, dtype=torch.float32):
    """ImageNet-normalised images are ~unit-variance, so N(0,1) is the right synthetic distribution
    (reference train_VIGOR.py:57-70)."""
    g = torch.Generator(device="cpu")
    g.manual_seed(10_000 + seed)
    grd = torch.randn((batch, 3) + tuple(ground_hw), generator=g).to(dtype)
    sat = torch.randn((batch, 3) + AERIAL_SHAPE, generator=g).to(dtype)
    return grd, sat


def synthetic_labels(batch: int, seed: int = 0, size: int = 512):
    """Compact synthetic training labels with the statistics of the reference dataset (reference datasets.py:142-166):
    gt [B, 1, size, size], a sigma-4 Gaussian at a random pixel, and each pair's orientation in degrees, a float64 [B]
    tensor in [0, 360).  `losses.orientation_labels(angles)` turns the angles into the bin weights and unit vectors that
    `losses.training_loss_from_labels` reads; `synthetic_ground_truth` expands the same draws into the dense maps."""
    g = torch.Generator().manual_seed(20_000 + seed)
    ys = torch.arange(size, dtype=torch.float32).view(size, 1)
    xs = torch.arange(size, dtype=torch.float32).view(1, size)
    gt = torch.zeros(batch, 1, size, size)
    angles = torch.zeros(batch, dtype=torch.float64)
    for b in range(batch):
        cy, cx = (torch.rand(2, generator=g) * (size - 64) + 32).tolist()
        gt[b, 0] = torch.exp(-((ys - cy) ** 2 + (xs - cx) ** 2) / (2.0 * 4.0 ** 2))
        angles[b] = float(torch.rand(1, generator=g)) * 360.0
    return gt, angles


def synthetic_ground_truth(batch: int, seed: int = 0, size: int = 512, n_bins: int = 20):
    """Synthetic training ground truth with the statistics of the reference dataset (reference datasets.py:142-166): a sigma-4 Gaussian at a random
    pixel, the same Gaussian split over two adjacent orientation bins, and a constant unit-vector orientation field.
    The dense form of `synthetic_labels` (same draws for the same seed)."""
    gt, angles = synthetic_labels(batch, seed, size)
    bin_weights, ori_vec = orientation_labels(angles, n_bins)
    gt_with_ori = gt * bin_weights[:, :, None, None]
    gt_orientation = ori_vec[:, :, None, None].expand(batch, 2, size, size).contiguous()
    return gt, gt_with_ori, gt_orientation
