"""Deterministic synthetic weights and inputs (there is no network for checkpoints or datasets).

`fill_deterministic` overwrites every tensor of a `state_dict` from a per-key seeded CPU generator, so two
models with the same state_dict keys (the reference's and ours) get bit-identical weights regardless of how
many random numbers their constructors consumed (SURVEY.md section 8(c) "Identical weights").  Scales are
He-style so activations keep O(1) magnitude through the 12-conv decoders and the 512x512 heatmap has a
well separated maximum (the reference's default init gives an almost flat heatmap, top-2 logit gap 8.6e-5,
which makes end-to-end argmax comparisons meaningless -- SURVEY.md section 7.3-4).
"""
from __future__ import annotations

import math
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
    poses = synthetic_poses(batch, seed, size)
    ys = torch.arange(size, dtype=torch.float32).view(size, 1)
    xs = torch.arange(size, dtype=torch.float32).view(1, size)
    gt = torch.zeros(batch, 1, size, size)
    for b in range(batch):
        cy, cx = poses[b, :2].tolist()
        gt[b, 0] = torch.exp(-((ys - cy) ** 2 + (xs - cx) ** 2) / (2.0 * 4.0 ** 2))
    return gt, poses[:, 2].clone()


def synthetic_poses(batch: int, seed: int = 0, size: int = 512):
    """The poses `synthetic_labels` draws for the same seed (same random sequence): a float64 [B, 3] CPU tensor of rows
    (row, col, angle_deg), the Gaussian's centre and the orientation in [0, 360).  `losses.training_loss_from_poses` builds
    the labels from them on the device."""
    g = torch.Generator().manual_seed(20_000 + seed)
    poses = torch.zeros(batch, 3, dtype=torch.float64)
    for b in range(batch):
        cy, cx = (torch.rand(2, generator=g) * (size - 64) + 32).tolist()
        poses[b] = torch.tensor([cy, cx, float(torch.rand(1, generator=g)) * 360.0], dtype=torch.float64)
    return poses


def synthetic_ground_truth(batch: int, seed: int = 0, size: int = 512, n_bins: int = 20):
    """Synthetic training ground truth with the statistics of the reference dataset (reference datasets.py:142-166): a sigma-4 Gaussian at a random
    pixel, the same Gaussian split over two adjacent orientation bins, and a constant unit-vector orientation field.
    The dense form of `synthetic_labels` (same draws for the same seed)."""
    gt, angles = synthetic_labels(batch, seed, size)
    bin_weights, ori_vec = orientation_labels(angles, n_bins)
    gt_with_ori = gt * bin_weights[:, :, None, None]
    gt_orientation = ori_vec[:, :, None, None].expand(batch, 2, size, size).contiguous()
    return gt, gt_with_ori, gt_orientation


def synthetic_mixture(batch: int, n_modes: int, H: int = 512, W: int = 512, seed: int = 0):
    """Multi-modal heatmaps, fp32 [B, 1, H, W] CPU, each summing to 1 like a softmax output: a mixture of `n_modes`
    isotropic Gaussians with random centres (anywhere in the map, edges included), widths sigma in [2, 12) and weights.
    The peaks are the planted location modes; the tails between them add many shallow ones."""
    g = torch.Generator().manual_seed(30_000 + seed)
    ys = torch.arange(H, dtype=torch.float64).view(H, 1)
    xs = torch.arange(W, dtype=torch.float64).view(1, W)
    out = torch.zeros(batch, 1, H, W)
    for b in range(batch):
        m = torch.zeros(H, W, dtype=torch.float64)
        for _ in range(n_modes):
            cy, cx = float(torch.rand(1, generator=g)) * (H - 1), float(torch.rand(1, generator=g)) * (W - 1)
            sigma = 2.0 + 10.0 * float(torch.rand(1, generator=g))
            w = 0.2 + float(torch.rand(1, generator=g))
            m += w * torch.exp(-(ys - cy) ** 2 / (2 * sigma ** 2)) * torch.exp(-(xs - cx) ** 2 / (2 * sigma ** 2))
        out[b, 0] = (m / m.sum()).float()
    return out


def synthetic_track(n_frames: int, batch: int = 1, H: int = 512, W: int = 512, seed: int = 0, sigma: float = 4.0):
    """A seeded sequence of heatmaps along a known trajectory, for the sequential location filter (`track_step`).

    Each of `batch` vehicles drives through a map at 3-6 map pixels per frame with a slowly turning heading.  Every frame's
    aerial crop is cut at an integer offset that puts the vehicle within 40 pixels of the crop's centre (a noisy position
    prior), with the translation-only crop data [1, 0, left, 0, 1, top].  The heatmap holds two isotropic Gaussians of
    width `sigma`: the true mode at the vehicle's position (peak 1) and a distractor at a random place at least
    min(100, max(H, W) / 4) pixels away (peak 1.5 on frames where it is stronger, about one in three from frame 1 on,
    else 0.5), plus a floor of 1e-6, normalised to sum 1.

    Returns a dict of CPU tensors: heatmap fp32 [T, B, 1, H, W]; motion float64 [T, B, 6], the true motion of each frame
    from the previous one (`models.track_motion`; frame 0: identity); truth float64 [T, B, 2] and distractor float64
    [T, B, 2], the (row, col) of both modes in crop pixels; strong bool [T, B], where the distractor has the higher peak."""
    from .models import track_motion

    rng = torch.Generator().manual_seed(40_000 + seed)
    rand = lambda: float(torch.rand(1, generator=rng))
    ys = torch.arange(H, dtype=torch.float64).view(H, 1)
    xs = torch.arange(W, dtype=torch.float64).view(1, W)
    heat = torch.empty(n_frames, batch, 1, H, W)
    motion = torch.zeros(n_frames, batch, 6, dtype=torch.float64)
    truth = torch.empty(n_frames, batch, 2, dtype=torch.float64)
    distractor = torch.empty(n_frames, batch, 2, dtype=torch.float64)
    strong = torch.zeros(n_frames, batch, dtype=torch.bool)

    def bump(cy, cx):
        return torch.exp(-((ys - cy) ** 2 + (xs - cx) ** 2) / (2 * sigma ** 2))

    far = min(100.0, max(H, W) / 4)                          # reachable from any vehicle position
    for b in range(batch):
        pos = [10_000.0 * rand(), 10_000.0 * rand()]              # (x, y) in map pixels
        heading = 2 * math.pi * rand()
        prev_crop = None
        for t in range(n_frames):
            if t:
                heading += 0.2 * (rand() - 0.5)
                speed = 3.0 + 3.0 * rand()
                step = (speed * math.cos(heading), speed * math.sin(heading))
                pos = [pos[0] + step[0], pos[1] + step[1]]
            left = math.floor(pos[0] - W / 2 + 80 * (rand() - 0.5))
            top = math.floor(pos[1] - H / 2 + 80 * (rand() - 0.5))
            crop = [1.0, 0.0, float(left), 0.0, 1.0, float(top)]
            motion[t, b] = torch.tensor(track_motion(prev_crop, crop, step) if t else [1.0, 0.0, 0.0, 0.0, 1.0, 0.0],
                                        dtype=torch.float64)
            prev_crop = crop
            cy, cx = pos[1] - top, pos[0] - left
            while True:
                dy, dx = rand() * (H - 1), rand() * (W - 1)
                if (dy - cy) ** 2 + (dx - cx) ** 2 >= far ** 2:
                    break
            strong[t, b] = t > 0 and rand() < 1 / 3
            m = bump(cy, cx) + (1.5 if strong[t, b] else 0.5) * bump(dy, dx) + 1e-6
            heat[t, b, 0] = (m / m.sum()).float()
            truth[t, b] = torch.tensor([cy, cx], dtype=torch.float64)
            distractor[t, b] = torch.tensor([dy, dx], dtype=torch.float64)
    return dict(heatmap=heat, motion=motion, truth=truth, distractor=distractor, strong=strong)
