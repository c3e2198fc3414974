"""CPU: host-side contract of the drop-in boundary -- state_dict keys, C-ABI symbols, loud failure without a GPU."""
import ctypes
import os
import re

import pytest
import torch

from ccvpe_b200 import cabi, models, specs
from ccvpe_b200.synthetic import fill_deterministic

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_cabi_library_loads_and_exports_every_declared_symbol():
    lib = cabi.load()
    assert lib.ccvpe_abi_version() == cabi.ABI_VERSION
    header = open(os.path.join(ROOT, "include", "ccvpe_b200.h")).read()
    declared = set(re.findall(r"\b(ccvpe_[a-z0-9_]+)\s*\(", header))
    declared.discard("ccvpe_igemm_desc")
    assert declared == set(cabi.EXPORTED_SYMBOLS)
    for name in declared:
        assert hasattr(lib, name), name


def test_igemm_desc_mirror_matches_c_layout():
    # LP64 layout of ccvpe_igemm_desc: 2 ptr, 15 int32 (+4 pad), 6 ptr, 4 int32, ptr, int32 (+4 pad); checked against
    # sizeof/offsetof of the C struct compiled from include/ccvpe_b200.h
    assert ctypes.sizeof(cabi.IgemmDesc) == 160
    assert (cabi.IgemmDesc.w_kn.offset, cabi.IgemmDesc.out.offset, cabi.IgemmDesc.backend.offset) == (80, 144, 152)


@pytest.mark.parametrize("ctor,n_rolls,sat_dim", [
    (lambda: models.CVM_VIGOR("cpu", True), 20, 1280),
    (lambda: models.CVM_VIGOR_ori_prior("cpu", 72.0, False), 20, 1280),
    (lambda: models.CVM_KITTI("cpu"), 16, 2048),
    (lambda: models.CVM_OxfordRobotCar("cpu"), 20, 1280),
])
def test_state_dict_contract(ctor, n_rolls, sat_dim):
    m = ctor()
    sd = m.state_dict()
    assert len(sd) == 818                                              # SURVEY section 8(b)
    head = [k for k in sd if not k.startswith(("grd_efficientnet", "sat_efficientnet"))]
    assert len(head) == 98
    assert tuple(sd["sat_feature_to_descriptors.1.weight"].shape) == (sat_dim, 5120)
    assert tuple(sd["deconv6.weight"].shape) == (sat_dim + 1, 1024, 2, 2)
    assert tuple(sd["deconv6_ori.weight"].shape) == (sat_dim + n_rolls, 1024, 2, 2)
    assert tuple(sd["conv1.2.weight"].shape) == (1, 16, 3, 3) and tuple(sd["conv1_ori.2.weight"].shape) == (2, 16, 3, 3)
    # round trip through a fresh instance (checkpoint compatibility)
    fill_deterministic(sd, seed=1)
    m2 = ctor()
    assert m2.load_state_dict(sd, strict=True).missing_keys == []


def test_no_cpu_fallback():
    m = models.CVM_VIGOR("cpu", True).eval()
    with pytest.raises(cabi.CcvpeError):
        with torch.no_grad():
            m(torch.zeros(1, 3, 320, 640), torch.zeros(1, 3, 512, 512))
    with pytest.raises(cabi.CcvpeError):
        models.CVM_VIGOR.decode_pose(torch.zeros(1, 1, 8, 8), torch.zeros(1, 2, 8, 8))
    with pytest.raises(cabi.CcvpeError):
        cabi.softmax_heatmap(torch.zeros(1, 8), torch.zeros(1, 8), torch.zeros(128))


def test_specs_match_reference_tables():
    assert specs.VIGOR.level_channels() == (1280, 640, 320, 160, 80, 40)
    assert specs.KITTI.level_channels() == (2048, 512, 256, 128, 128, 32)
    assert specs.OXFORD.window_offset(1280, 224) == 528 and specs.OXFORD.window_len(40, 7) == 7   # models.py:1094
    assert specs.loc_roll_indices(specs.VIGOR, 72.0) == list(range(-4, 5))                          # models.py:489
    assert specs.loc_roll_indices(specs.KITTI, None) == list(range(16))


def test_pad_k_blocks_layout_rule():
    """w_nk K padding documented in include/ccvpe_b200.h and used by the kernels (tc_block_width): block width 16 if
    K <= 16, 32 if K <= 32, else 64; zero filled.  Each source of a two-source layout is padded by its own width."""
    for K, padded in [(16, 16), (24, 32), (40, 64), (80, 128), (112, 128), (192, 192), (320, 320), (8, 16),
                      (32, 32), (33, 64), (63, 64), (64, 64)]:
        w = torch.arange(3 * K, dtype=torch.float32).reshape(3, K) + 1.0
        out = cabi.pad_k_blocks(w)
        assert out.dtype == torch.bfloat16 and tuple(out.shape) == (3, padded), (K, out.shape)
        assert torch.equal(out[:, :K].float(), w.to(torch.bfloat16).float())
        assert float(out[:, K:].abs().sum()) == 0.0
    # two sources of 40 + 24 channels over 9 taps -> 64 + 32 per tap
    rows = torch.arange(2 * 9 * 64, dtype=torch.float32).reshape(2, 9, 64) + 1.0
    out = cabi.w_nk_layout(rows, [40, 24])
    assert out.dtype == torch.bfloat16 and tuple(out.shape) == (2, 9, 96), out.shape
    assert torch.equal(out[:, :, :40].float(), rows[:, :, :40].to(torch.bfloat16).float())
    assert torch.equal(out[:, :, 64:88].float(), rows[:, :, 40:].to(torch.bfloat16).float())
    assert float(out[:, :, 40:64].abs().sum()) == 0.0 and float(out[:, :, 88:].abs().sum()) == 0.0


def test_cuda_graph_cache_is_dropped_when_weights_change():
    """set_cuda_graph keeps one graph per input signature; anything that can move or change weights must drop them."""
    m = models.CVM_VIGOR("cpu", True).eval()
    assert m._graphs[0] is None                                  # eager by default
    m.set_cuda_graph(True)
    m._graphs[0]["sentinel"] = object()
    m.load_state_dict(m.state_dict())
    assert m._graphs[0] == {}
    m._graphs[0]["sentinel"] = object()
    m.set_precision("bf16")
    assert m._graphs[0] == {}
    m._graphs[0]["sentinel"] = object()
    m.float()
    assert m._graphs[0] == {}
    m.set_cuda_graph(False)
    assert m._graphs[0] is None
    with pytest.raises(cabi.CcvpeError):                         # still no CPU path, graph mode or not
        m(torch.zeros(1, 3, 320, 640), torch.zeros(1, 3, 512, 512))
