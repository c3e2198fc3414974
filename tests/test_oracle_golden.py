"""CPU: the oracle restatement reproduces the fixtures generated from the UNMODIFIED reference
(oracle/make_golden.py).  Runs everywhere (no reference checkout, no GPU needed)."""
import os

import numpy as np
import pytest
import torch

from helpers import GOLDEN_CONFIGS, GOLDEN_THREADS, build_model, check_against_golden, config_inputs, oracle_forward
from oracle import ccvpe_oracle as orc

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture
def golden_threads():
    saved = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(saved)


@pytest.mark.parametrize("name", sorted(GOLDEN_CONFIGS))
def test_oracle_matches_reference_fixture(golden_threads, name):
    variant, shape_key, noise, circular, batch, wseed, iseed = GOLDEN_CONFIGS[name]
    golden = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    model = build_model(variant, noise, circular, wseed)
    grd, sat = config_inputs(name)
    out = oracle_forward(model, variant, noise, grd, sat)
    # fp32 CPU at the fixtures' thread count; a different CPU may still round differently: tolerance 1e-5 of max-abs per tensor
    check_against_golden(out, golden, tol=1e-5)
    pose = orc.pose_decode(out[1].numpy(), out[2].numpy())
    assert pose["idx"].tolist() == golden["pose.idx"].tolist()          # bit-exact indices
    assert pose["rc"].tolist() == golden["pose.rc"].tolist()
    np.testing.assert_allclose(pose["angle"], golden["pose.angle"], rtol=0, atol=1e-2)
    assert pose["valid"].tolist() == golden["pose.valid"].tolist()


def loss_inputs():
    """Seeded scores / labels / logits / orientation fields for the oracle losses (64x64 maps, batch 2-3)."""
    from ccvpe_b200.synthetic import synthetic_ground_truth
    g = torch.Generator().manual_seed(5)
    s = torch.rand(3, 20 * 64, generator=g) * 2 - 1
    lab = torch.rand(3, 20 * 64, generator=g) * (torch.rand(3, 20 * 64, generator=g) > 0.9)
    logits = torch.randn(2, 4096, generator=g)
    soft = torch.softmax(torch.randn(2, 4096, generator=g), dim=1)
    gt, gwo, gor = synthetic_ground_truth(2, seed=1, size=64)
    ori = torch.nn.functional.normalize(torch.randn(2, 2, 64, 64, generator=g), dim=1)
    outs = [logits, None, ori] + [torch.rand(2, 20, 64 // k, 64 // k, generator=g) * 2 - 1 for k in (64, 32, 16, 8, 4, 2)]
    return s, lab, logits, soft, ori, gt, gwo, gor, outs


def oracle_losses():
    s, lab, logits, soft, ori, gt, gwo, gor, outs = loss_inputs()
    return {"infonce": orc.infonce_loss(s, lab), "cross_entropy": orc.cross_entropy_loss(logits, soft),
            "orientation": orc.orientation_loss(ori, gor, gt), "training": orc.training_loss(outs, gt, gwo, gor)}


def test_oracle_losses_match_stored_values():
    """The oracle's restatement of the original losses.py:4-29 and of the loss combination of train_VIGOR.py:120-146 (what
    tests/test_gpu_train.py checks the fused CUDA losses against) reproduces the values stored in
    tests/golden/oracle_losses.npz.  The values were recorded from the oracle as it stood when it was last compared, bit for
    bit, with the original losses.py; the tolerance covers summation-order differences between CPUs."""
    golden = np.load(os.path.join(GOLDEN_DIR, "oracle_losses.npz"))
    for name, value in oracle_losses().items():
        np.testing.assert_allclose(value.item(), golden[name], rtol=1e-6, err_msg=name)


def test_pose_decode_edge_cases():
    """first-occurrence ties, plateau, extremes, invalid (|cos|>1) -- semantics of train_VIGOR.py:297-316."""
    H = W = 8
    heat = np.zeros((5, 1, H, W), np.float32)
    ori = np.zeros((5, 2, H, W), np.float32)
    heat[0, 0, 3, 4] = heat[0, 0, 5, 1] = 1.0          # tie -> first in raster order
    heat[1] = 0.25                                      # plateau -> index 0
    heat[2, 0, 7, 7] = 2.0                              # last element
    heat[3, 0, 0, 0] = 2.0
    heat[4, 0, 2, 2] = 1.0
    ori[0, :, 3, 4] = (0.0, -1.0)
    ori[1, :, 0, 0] = (1.0, 0.0)
    ori[2, :, 7, 7] = (-1.0, 0.0)
    ori[3, :, 0, 0] = (np.float32(0.6), np.float32(0.8))
    ori[4, :, 2, 2] = (1.5, 0.0)                        # invalid
    p = orc.pose_decode(heat, ori)
    assert p["idx"].tolist() == [3 * W + 4, 0, 63, 0, 2 * W + 2]
    assert p["valid"].tolist() == [1, 1, 1, 1, 0]
    np.testing.assert_allclose(p["angle"][:4], [270.0, 0.0, 180.0, np.degrees(np.arccos(np.float64(np.float32(0.6))))])
    assert np.isnan(p["angle"][4])
