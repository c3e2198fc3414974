"""CPU ORACLE -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

A CPU restatement (torch-CPU / numpy, fp32 by default, fp64 on request) of the post-encoder hot path of
tudelft-iv/CCVPE, i.e. what `CVM_VIGOR / CVM_VIGOR_ori_prior / CVM_KITTI / CVM_OxfordRobotCar.forward` do
after the two EfficientNet-B0 encoders, plus the host-side argmax pose decode of the scripts.  Every function
cites the reference file:line it follows.  The arithmetic of conv / conv-transpose / softmax lives in ATen
(third party, torch 2.11.0 in this image; the reference pins no version) exactly as it does for the reference.

Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference` leg may import
this file, and only as the checker / the timed CPU baseline -- never as (part of) the product path.

PARITY PINNING: the reference ships no tests or golden vectors for this path (SURVEY.md section 4), so the
oracle is pinned against outputs of the reference itself executed in the authoring container:
`oracle/make_golden.py` imports the unmodified reference (via `oracle/ref_shim.py`), runs it on seeded
weights/inputs and commits digests + samples of all nine outputs to `tests/golden/*.npz`;
`tests/test_oracle_golden.py` checks this file against those fixtures, and its losses against values stored in
`tests/golden/oracle_losses.npz`.

The op ORDER deliberately mirrors the reference (roll -> window -> norm -> mul -> sum -> cat per orientation)
so that timing this file on host cores is a fair stand-in for the reference's CPU forward.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
from torch.nn import functional as F

Tensor = torch.Tensor

# ---------------------------------------------------------------------------------------------
# Per-class constants (reference models.py; SURVEY.md section 8 table)
# ---------------------------------------------------------------------------------------------
VARIANTS: Dict[str, dict] = {
    # CVM_VIGOR models.py:186-314 -- 20 orientations, roll strides 64..2, window = first L channels
    "vigor": dict(n_rolls=20, strides=(64, 32, 16, 8, 4, 2), centred=False),
    # CVM_VIGOR_ori_prior models.py:484-623 -- same strides; loc rolls limited to [-k, k]
    "vigor_prior": dict(n_rolls=20, strides=(64, 32, 16, 8, 4, 2), centred=False),
    # CVM_KITTI models.py:788-920 -- 16 orientations, strides 128,64,32,16,8,8
    "kitti": dict(n_rolls=16, strides=(128, 64, 32, 16, 8, 8), centred=False),
    # CVM_OxfordRobotCar models.py:1087-1215 -- 20 orientations, centred window (:1094)
    "oxford": dict(n_rolls=20, strides=(64, 32, 16, 8, 4, 2), centred=True),
}


def _roll_list(variant: str, ori_noise: Optional[float]) -> List[int]:
    """Orientation indices used by the localisation branch (models.py:191 / :489 / :793 / :1092)."""
    if variant == "vigor_prior":
        k = int(ori_noise / 18)
        return list(range(-k, k + 1))
    return list(range(VARIANTS[variant]["n_rolls"]))


# ---------------------------------------------------------------------------------------------
# a1  ground descriptor heads   (models.py:22-31, 57-97, 152-157)
# ---------------------------------------------------------------------------------------------
def grd_descriptor(feature_volume: Tensor, w1: Tensor, b1: Tensor, w2: Tensor, b2: Tensor) -> Tensor:
    """1x1 conv 1280->c, permute (B,C,H,W)->(B,H,W,C), 1x1 conv over the height axis H->1, flatten.

    Result index is w*c + ch (azimuth major) which is what makes a channel roll a rotation."""
    y = F.conv2d(feature_volume, w1, b1)              # [B, c, H, W]
    y = y.permute(0, 2, 3, 1)                         # [B, H, W, c]   (H is now the "channel" axis)
    y = F.conv2d(y, w2, b2)                           # [B, 1, W, c]
    return y.flatten(1)                               # [B, W*c]


def grd_descriptors(feature_volume: Tensor, sd: Dict[str, Tensor]) -> List[Tensor]:
    return [
        grd_descriptor(
            feature_volume,
            sd["grd_feature_to_descriptor%d.0.weight" % lvl], sd["grd_feature_to_descriptor%d.0.bias" % lvl],
            sd["grd_feature_to_descriptor%d.2.weight" % lvl], sd["grd_feature_to_descriptor%d.2.bias" % lvl],
        )
        for lvl in range(1, 7)
    ]


# ---------------------------------------------------------------------------------------------
# a3  aerial cell descriptors   (models.py:102-104, 173-184)
# ---------------------------------------------------------------------------------------------
def sat_cell_descriptors(sat_feature_volume: Tensor, weight: Tensor, bias: Tensor) -> Tensor:
    """8x8 grid of cells, each cell (C, H/8, W/8) flattened in (c, dh, dw) order through one Linear."""
    rows = []
    for row_chunk in torch.chunk(sat_feature_volume, 8, dim=2):
        cells = []
        for cell in torch.chunk(row_chunk, 8, dim=3):
            cells.append(F.linear(cell.flatten(1), weight, bias)[:, :, None, None])
        rows.append(torch.cat(cells, dim=3))
    return torch.cat(rows, dim=2)                     # [B, D, 8, 8]


# ---------------------------------------------------------------------------------------------
# a4/a5  rolled cosine matching   (models.py:186-202 and the 23 sibling loops)
# ---------------------------------------------------------------------------------------------
def match_level(x: Tensor, g: Tensor, rolls: Sequence[int], stride: int, centred: bool) -> Tensor:
    """scores[b,i,p] = <g_b, window_i(x)_p> / (||window_i(x)_p|| * ||g_b||), no epsilon (models.py:196).

    window_i = channels [o, o+L) of roll(x, -i*stride, dim=1); o = 0, or int(C/2 - L/2) for the centred
    variant (models.py:1094)."""
    B, C, H, W = x.shape
    L = g.shape[1]
    g_map = g[:, :, None, None].repeat(1, 1, H, W)                      # models.py:159-164
    g_norm = torch.norm(g_map, p="fro", dim=1, keepdim=True)            # models.py:189
    lo, hi = (int(C / 2 - L / 2), int(C / 2 + L / 2)) if centred else (0, L)
    per_roll = []
    for i in rolls:
        rolled = torch.roll(x, shifts=-i * stride, dims=1)
        window = rolled[:, lo:hi]
        w_norm = torch.norm(window, p="fro", dim=1, keepdim=True)
        per_roll.append(torch.sum(g_map * window, dim=1, keepdim=True) / (w_norm * g_norm))
    return torch.cat(per_roll, dim=1)                                   # [B, len(rolls), H, W]


# ---------------------------------------------------------------------------------------------
# a6  L2 normalisation over channels   (models.py:33-40)
# ---------------------------------------------------------------------------------------------
def l2_normalize(x: Tensor) -> Tensor:
    return F.normalize(x, p=2, dim=1)                                   # x / max(||x||, 1e-12)


# ---------------------------------------------------------------------------------------------
# a7-a9  one Localization-Matching-Upsampling step   (models.py:205-209 etc.)
# ---------------------------------------------------------------------------------------------
def upsample_block(x: Tensor, skip: Optional[Tensor], sd: Dict[str, Tensor], deconv: str, conv: str) -> Tensor:
    """ConvTranspose2d(k2,s2) -> cat(skip) -> conv3x3 -> ReLU -> conv3x3   (models.py:42-47, 207-209)."""
    x = F.conv_transpose2d(x, sd[deconv + ".weight"], sd[deconv + ".bias"], stride=2)
    if skip is not None:
        x = torch.cat([x, skip], dim=1)
    x = F.relu(F.conv2d(x, sd[conv + ".0.weight"], sd[conv + ".0.bias"], padding=1))
    return F.conv2d(x, sd[conv + ".2.weight"], sd[conv + ".2.bias"], padding=1)


# ---------------------------------------------------------------------------------------------
# a10  heatmap softmax   (models.py:319-320)
# ---------------------------------------------------------------------------------------------
def softmax_heatmap(logits_map: Tensor) -> Tuple[Tensor, Tensor]:
    flat = logits_map.flatten(1)
    return flat, torch.softmax(flat, dim=-1).reshape(logits_map.shape)


# ---------------------------------------------------------------------------------------------
# whole post-encoder path   (models.py:152-343 / :450-652 / :753-950 / :1052-1244)
# ---------------------------------------------------------------------------------------------
def forward_post_encoder(variant: str, sd: Dict[str, Tensor], grd_feature_volume: Tensor,
                         sat_feature_volume: Tensor, multiscale_sat: Sequence[Tensor],
                         ori_noise: Optional[float] = None, intermediates: Optional[dict] = None):
    """Returns the reference's 9-tuple (models.py:343)."""
    spec = VARIANTS[variant]
    skips = [multiscale_sat[i] for i in (15, 10, 4, 2, 0)]              # models.py:167-171
    g = grd_descriptors(grd_feature_volume, sd)
    x = sat_cell_descriptors(sat_feature_volume, sd["sat_feature_to_descriptors.1.weight"],
                             sd["sat_feature_to_descriptors.1.bias"])
    loc_rolls = _roll_list(variant, ori_noise)
    all_rolls = list(range(spec["n_rolls"]))

    scores = []
    # bottleneck level
    s_loc = match_level(x, g[0], loc_rolls, spec["strides"][0], spec["centred"])
    s_full = s_loc if variant != "vigor_prior" else match_level(x, g[0], all_rolls, spec["strides"][0],
                                                                spec["centred"])   # models.py:501-511
    scores.append(s_full)
    x_hat_1 = l2_normalize(x)
    x_bottleneck = x
    if intermediates is not None:
        intermediates["g"] = g
        intermediates["x"] = [x]
    x = torch.cat([s_loc.max(dim=1, keepdim=True)[0], x_hat_1], dim=1)
    for lvl in range(2, 7):                                             # levels 2..6, models.py:207-315
        x = upsample_block(x, skips[lvl - 2], sd, "deconv%d" % (8 - lvl), "conv%d" % (8 - lvl))
        if intermediates is not None:
            intermediates["x"].append(x)
        s = match_level(x, g[lvl - 1], loc_rolls, spec["strides"][lvl - 1], spec["centred"])
        scores.append(s)
        x = torch.cat([s.max(dim=1, keepdim=True)[0], l2_normalize(x)], dim=1)
    x = upsample_block(x, None, sd, "deconv1", "conv1")                 # models.py:316-317
    logits_flat, heatmap = softmax_heatmap(x)

    # orientation decoder (models.py:322-341) -- no matching inside
    o = torch.cat([s_full, l2_normalize(x_bottleneck)], dim=1)
    for lvl in range(2, 7):
        o = upsample_block(o, skips[lvl - 2], sd, "deconv%d_ori" % (8 - lvl), "conv%d_ori" % (8 - lvl))
    o = upsample_block(o, None, sd, "deconv1_ori", "conv1_ori")
    if intermediates is not None:
        intermediates["ori_raw"] = o
    o = F.normalize(o, p=2, dim=1)
    return (logits_flat, heatmap, o, *scores)


# ---------------------------------------------------------------------------------------------
# a13  host pose decode   (train_VIGOR.py:290-326 and its eight copies)
# ---------------------------------------------------------------------------------------------
def pose_decode(heatmap: np.ndarray, ori: np.ndarray):
    """heatmap [B,1,H,W], ori [B,2,H,W] (numpy).  Returns dict of arrays:
    idx int64[B] (first-occurrence argmax over probabilities), rc int32[B,2], cs float32[B,2],
    angle float64[B] in degrees [0,360) (NaN where invalid), valid uint8[B]."""
    B = heatmap.shape[0]
    out = dict(idx=np.zeros(B, np.int64), rc=np.zeros((B, 2), np.int32), cs=np.zeros((B, 2), np.float32),
               angle=np.full(B, np.nan, np.float64), valid=np.zeros(B, np.uint8))
    for b in range(B):
        cur = heatmap[b]
        loc = np.unravel_index(cur.argmax(), cur.shape)                 # train_VIGOR.py:297
        out["idx"][b] = loc[1] * cur.shape[2] + loc[2]
        out["rc"][b] = (loc[1], loc[2])
        cos_pred, sin_pred = ori[b, :, loc[1], loc[2]]                  # train_VIGOR.py:310
        out["cs"][b] = (cos_pred, sin_pred)
        if np.abs(cos_pred) <= 1 and np.abs(sin_pred) <= 1:             # train_VIGOR.py:311
            a = math.acos(cos_pred)
            out["angle"][b] = math.degrees(-a) % 360 if sin_pred < 0 else math.degrees(a)
            out["valid"][b] = 1
    return out


# ---------------------------------------------------------------------------------------------
# full forward incl. encoders -- used only as the timed CPU baseline (bench.py cpu_baseline / --impl reference)
# ---------------------------------------------------------------------------------------------
def forward_full(variant: str, sd: Dict[str, Tensor], grd_encoder, sat_encoder, grd: Tensor, sat: Tensor,
                 ori_noise: Optional[float] = None, intermediates: Optional[dict] = None):
    """Encoders are the caller's torch modules (the encoders stay PyTorch in reference and product alike)."""
    fg = grd_encoder.extract_features(grd)                              # models.py:151
    fs, multi = sat_encoder.extract_features_multiscale(sat)            # models.py:166
    return forward_post_encoder(variant, sd, fg, fs, multi, ori_noise, intermediates)


# ---------------------------------------------------------------------------------------------
# training losses   (losses.py:4-29) and their combination (train_VIGOR.py:120-146) -- used with torch autograd as the
# reference for the loss values and for every gradient of the training step (tests/test_gpu_train.py)
# ---------------------------------------------------------------------------------------------
def infonce_loss(scores: Tensor, labels: Tensor, temperature: float = 0.1) -> Tensor:
    exp_scores = torch.exp(scores / temperature)                         # losses.py:13
    mask = labels > 1e-2                                                 # losses.py:14
    denominator = torch.sum(exp_scores, dim=1, keepdim=True)             # losses.py:16
    inner = torch.log(torch.masked_select(exp_scores / denominator, mask))
    w = torch.masked_select(labels, mask)
    return -torch.sum(inner * w) / torch.sum(w)                          # losses.py:18


def cross_entropy_loss(logits: Tensor, labels: Tensor) -> Tensor:
    return -torch.sum(labels * F.log_softmax(logits, dim=1)) / logits.size()[0]      # losses.py:24


def orientation_loss(ori: Tensor, gt_orientation: Tensor, gt: Tensor) -> Tensor:
    return torch.sum(torch.sum(torch.square(gt_orientation - ori), dim=1, keepdim=True) * gt) / ori.size()[0]   # losses.py:29


def training_loss(outputs, gt: Tensor, gt_with_ori: Tensor, gt_orientation: Tensor, weight_infonce: float = 1e4,
                  weight_ori: float = 1e1) -> Tensor:
    """train_VIGOR.py:120-146."""
    gt_flattened = torch.flatten(gt, start_dim=1)
    gt_flattened = gt_flattened / torch.sum(gt_flattened, dim=1, keepdim=True)
    loss_ori = orientation_loss(outputs[2], gt_orientation, gt)
    nce = 0
    for scores, k in zip(outputs[3:9], (64, 32, 16, 8, 4, 2)):
        gt_b = F.max_pool2d(gt_with_ori, k, stride=k)
        nce = nce + infonce_loss(torch.flatten(scores, start_dim=1), torch.flatten(gt_b, start_dim=1))
    loss_ce = cross_entropy_loss(outputs[0], gt_flattened)
    return loss_ce + weight_infonce * nce / 6 + weight_ori * loss_ori
