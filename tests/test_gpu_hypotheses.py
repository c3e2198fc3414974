"""Pose hypotheses (`decoder.decode_hypotheses`, C ABI `ccvpe_pose_hypotheses`): the k strongest mutually exclusive
location modes of each heatmap, their probability mass and orientation.

`reference` below is the semantics in plain NumPy.  The device output must equal it exactly in idx, rc, value, count, cs
and valid, and in mass to within one float32 ulp of the float64 sum rounded once.  The angle must equal `decode_pose`'s
rule at the same pixel bit for bit (checked by decoding the (cos, sin) pairs as 1x1 maps); against the reference's
`math.acos` it is held to 1e-9 degrees, as `decode_pose`'s own tests do, because CUDA's and the C library's acos may
differ in the last bit."""
import ctypes
import math

import numpy as np
import pytest
import torch
from torch.nn import functional as F

from ccvpe_b200 import cabi, models
from ccvpe_b200.decoder import decode_hypotheses, decode_pose
from ccvpe_b200.synthetic import synthetic_mixture
from helpers import GOLDEN_CONFIGS, build_model, config_inputs

KEYS = ("idx", "rc", "value", "mass", "cs", "angle", "valid", "count")
NAN, INF = float("nan"), float("inf")


# ---------------------------------------------------------------------------------------------------------------------
# NumPy reference
# ---------------------------------------------------------------------------------------------------------------------
def reference(h, ori, k, radius):
    """One pair: h float32 [H, W], ori float32 [2, H, W].  Returns the outputs of `decode_hypotheses` for that pair."""
    H, W = h.shape
    out = dict(idx=np.full(k, -1, np.int64), rc=np.full((k, 2), -1, np.int32), value=np.full(k, np.nan, np.float32),
               mass=np.full(k, np.nan, np.float32), cs=np.full((k, 2), np.nan, np.float32),
               angle=np.full(k, np.nan, np.float64), valid=np.zeros(k, np.uint8), count=0)
    if np.isnan(h).any():
        return out
    padded = np.pad(h, 1, constant_values=-np.inf)          # out-of-bounds neighbours never disqualify a mode
    mode = np.ones((H, W), bool)
    for di in (-1, 0, 1):
        for dj in (-1, 0, 1):
            if di or dj:
                mode &= h >= padded[1 + di:1 + di + H, 1 + dj:1 + dj + W]
    cand = np.flatnonzero(mode)
    order = cand[np.lexsort((cand, -h.reshape(-1)[cand]))]  # value descending, then the smaller flat index
    claimed = np.zeros((H, W), bool)
    h64 = h.astype(np.float64)
    t = 0
    for p in order:
        if t == k:
            break
        i0, j0 = divmod(int(p), W)
        if claimed[i0, j0]:
            continue
        ia, ib, ja, jb = max(i0 - radius, 0), min(i0 + radius, H - 1) + 1, max(j0 - radius, 0), min(j0 + radius, W - 1) + 1
        ii, jj = np.ogrid[ia:ib, ja:jb]
        disc = (ii - i0) ** 2 + (jj - j0) ** 2 <= radius * radius
        box = claimed[ia:ib, ja:jb]
        with np.errstate(invalid="ignore"):                 # +inf and -inf in one disc: NaN mass
            out["mass"][t] = np.float32(h64[ia:ib, ja:jb][disc & ~box].sum())
        box |= disc
        out["idx"][t], out["rc"][t], out["value"][t] = p, (i0, j0), h[i0, j0]
        c, s = ori[:, i0, j0]
        out["cs"][t] = (c, s)
        if abs(c) <= 1 and abs(s) <= 1:                     # decode_pose's rule (reference train_VIGOR.py:311)
            a = math.acos(c)
            out["angle"][t] = math.degrees(-a) % 360 if s < 0 else math.degrees(a)
            out["valid"][t] = 1
        t += 1
    out["count"] = t
    return out


def check_pair(got, ref, where=""):
    """got: the device outputs of one pair as NumPy arrays."""
    assert int(got["count"]) == ref["count"], where
    for key in ("idx", "rc", "valid"):
        assert np.array_equal(got[key], ref[key]), (where, key, got[key], ref[key])
    for key in ("value", "cs"):                             # bit for bit (the NaN of an empty slot included)
        assert np.array_equal(got[key].view(np.uint32), ref[key].view(np.uint32)), (where, key, got[key], ref[key])
    m, mr = got["mass"].astype(np.float64), ref["mass"].astype(np.float64)
    finite = np.isfinite(mr)
    assert np.array_equal(m[~finite], mr[~finite], equal_nan=True), (where, "mass", m, mr)
    ulp = np.spacing(np.abs(ref["mass"][finite])).astype(np.float64)
    assert (np.abs(m[finite] - mr[finite]) <= ulp).all(), (where, "mass", m, mr)
    np.testing.assert_allclose(got["angle"], ref["angle"], rtol=0, atol=1e-9, equal_nan=True, err_msg=where)


def run(heat, ori, k, radius):
    out = decode_hypotheses(heat, ori, k, radius)
    torch.cuda.synchronize()
    return {key: v.cpu().numpy() for key, v in out.items()}


def pair(out, b):
    return {key: out[key][b] for key in KEYS}


def check_batch(heat, ori, k, radius, name):
    """Device vs reference for every pair; angle and valid vs decode_pose's rule bit for bit; k = 1 vs decode_pose."""
    dev = torch.device("cuda:0")
    got = run(heat.to(dev), ori.to(dev), k, radius)
    h, o = heat.numpy(), ori.numpy()
    for b in range(heat.shape[0]):
        check_pair(pair(got, b), reference(h[b, 0], o[b], k, radius), "%s pair %d" % (name, b))
    # angle / valid: decode_pose applied to each hypothesis's (cos, sin) as a 1x1 map
    cs = torch.from_numpy(got["cs"].reshape(-1, 2)).view(-1, 2, 1, 1).to(dev)
    pose = decode_pose(torch.zeros(cs.shape[0], 1, 1, 1, device=dev), cs)
    filled = got["idx"].reshape(-1) >= 0
    assert np.array_equal(got["angle"].reshape(-1)[filled].view(np.uint64),
                          pose["angle"].cpu().numpy()[filled].view(np.uint64)), name
    assert np.array_equal(got["valid"].reshape(-1)[filled], pose["valid"].cpu().numpy()[filled]), name
    # k = 1 equals decode_pose bit for bit on every NaN-free map
    ok = ~torch.isnan(heat).flatten(1).any(1).numpy()
    one = run(heat.to(dev), ori.to(dev), 1, radius)
    ref = {key: v.cpu().numpy() for key, v in decode_pose(heat.to(dev), ori.to(dev)).items()}
    assert np.array_equal(one["idx"][ok, 0], ref["idx"][ok]), name
    assert np.array_equal(one["rc"][ok, 0], ref["rc"][ok]), name
    assert np.array_equal(one["cs"][ok, 0].view(np.uint32), ref["cs"][ok].view(np.uint32)), name
    assert np.array_equal(one["angle"][ok, 0].view(np.uint64), ref["angle"][ok].view(np.uint64)), name
    assert np.array_equal(one["valid"][ok, 0], ref["valid"][ok]), name
    return got


def unit_field(B, H, W, seed):
    ori = F.normalize(torch.randn(B, 2, H, W, generator=torch.Generator().manual_seed(seed)), dim=1)
    ori.view(B, 2, -1)[:, 0, ::97] = 1.5                    # some invalid orientations (|cos| > 1)
    return ori


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the reference on hand-worked maps, and every refusal
# ---------------------------------------------------------------------------------------------------------------------
def _ori(H, W):
    ori = np.zeros((2, H, W), np.float32)
    ori[0] = 1.0
    return ori


def test_reference_ties_go_to_the_smaller_flat_index():
    """Two equal peaks: the first in row-major order comes first (the last-occurrence rule would give [9, 1])."""
    h = np.zeros((3, 4), np.float32)
    h[0, 1] = h[2, 1] = 0.5
    ref = reference(h, _ori(3, 4), 2, 0)
    assert ref["idx"].tolist() == [1, 9] and ref["count"] == 2


def test_reference_claim_skips_modes_inside_an_earlier_disc():
    """Peaks at columns 0, 3 and 7 of one row.  r = 3: the peak at 3 is claimed by the one at 0 (distance 3 <= r), the
    one at 7 is not: hypotheses [0, 7] (a rule that claimed only other modes' pixels or used r - 1 would give 3)."""
    h = np.zeros((1, 9), np.float32)
    h[0, [0, 3, 7]] = [0.5, 0.3, 0.2]
    ref = reference(h, _ori(1, 9), 4, 3)
    assert ref["idx"][:2].tolist() == [0, 7]
    # 7's disc covers columns 4..8; columns 4..6 are fresh; column 3 is the first hypothesis's
    assert ref["mass"][:2].tolist() == [np.float32(0.8), np.float32(0.2)]
    # next after 7: the zero plateau is claimed everywhere (columns 0..8), so nothing is left
    assert ref["count"] == 2


def test_reference_mass_counts_only_pixels_no_earlier_disc_claimed():
    """3x5 map of ones with peaks 4 at (1, 1) and 2 at (1, 3), r = 1 (5-pixel plus-shaped discs).  The discs share (1, 2):
    the first takes it, so the masses are 1 + 1 + 4 + 1 + 1 = 8 and 1 + 2 + 1 + 1 = 5 (counting it twice would give 6).
    Every other pixel touches a peak, so there are exactly two modes."""
    h = np.ones((3, 5), np.float32)
    h[1, 1], h[1, 3] = 4, 2
    ref = reference(h, _ori(3, 5), 8, 1)
    assert ref["count"] == 2 and ref["idx"].tolist() == [6, 8] + [-1] * 6
    assert ref["mass"][:2].tolist() == [8.0, 5.0] and np.isnan(ref["mass"][2:]).all()


def test_reference_plateau_modes_and_nan_and_inf():
    const = np.full((2, 3), 0.25, np.float32)
    ref = reference(const, _ori(2, 3), 8, 0)                 # every pixel is a mode, r = 0 claims one pixel each
    assert ref["count"] == 6 and ref["idx"][:6].tolist() == list(range(6)) and ref["idx"][6] == -1
    assert np.isnan(ref["mass"][6]) and np.isnan(ref["value"][6]) and ref["valid"][6] == 0
    ninf = np.full((2, 2), -np.inf, np.float32)
    assert reference(ninf, _ori(2, 2), 1, 0)["idx"].tolist() == [0]
    h = np.zeros((2, 2), np.float32)
    h[1, 1] = np.nan
    assert reference(h, _ori(2, 2), 4, 1)["count"] == 0
    h[1, 1] = np.inf
    ref = reference(h, _ori(2, 2), 4, 0)
    assert ref["idx"][0] == 3 and ref["mass"][0] == np.inf


def _bind_args(B=2, H=16, W=24, k=4, **over):
    a = dict(heatmap=torch.zeros(B, 1, H, W), ori=torch.zeros(B, 2, H, W), k=k, radius=3)
    k = k if isinstance(k, int) and 1 <= k <= 64 else 4
    a.update(idx=torch.zeros(B, k, dtype=torch.int64), rc=torch.zeros(B, k, 2, dtype=torch.int32),
             value=torch.zeros(B, k), mass=torch.zeros(B, k), cs=torch.zeros(B, k, 2),
             angle=torch.zeros(B, k, dtype=torch.float64), valid=torch.zeros(B, k, dtype=torch.uint8),
             count=torch.zeros(B, dtype=torch.int32))
    a.update(over)
    return a


@pytest.mark.parametrize("over,msg", [
    (dict(k=0), "k must be"), (dict(k=65), "k must be"), (dict(k=2.0), "k must be"), (dict(k=True), "k must be"),
    (dict(radius=-1), "radius must be"), (dict(radius=32768), "radius must be"), (dict(radius=1.5), "radius must be"),
    (dict(heatmap=torch.zeros(2, 1, 16, 24, dtype=torch.float64)), "heatmap must be a float32"),
    (dict(heatmap=torch.zeros(2, 16, 24)), "heatmap must have shape"),
    (dict(heatmap=torch.zeros(2, 2, 16, 24)), "heatmap must have shape"),
    (dict(heatmap=torch.zeros(2, 1, 24, 16).transpose(2, 3)), "heatmap must be contiguous"),
    (dict(heatmap=torch.zeros(0, 1, 16, 24)), "0 < B"),
    (dict(heatmap=torch.zeros(2, 1, 8, 60000)), "does not fit"),
    (dict(ori=torch.zeros(2, 2, 16, 25)), "ori must have shape"),
    (dict(ori=torch.zeros(2, 2, 16, 24).to(torch.bfloat16)), "ori must be a float32"),
    (dict(idx=torch.zeros(2, 4, dtype=torch.int32)), "idx must be"),
    (dict(idx=torch.zeros(2, 5, dtype=torch.int64)), "idx must be"),
    (dict(rc=torch.zeros(2, 4, 2, dtype=torch.int64)), "rc must be"),
    (dict(rc=torch.zeros(2, 2, 4, dtype=torch.int32).transpose(1, 2)), "rc must be"),
    (dict(value=torch.zeros(2, 4, dtype=torch.float64)), "value must be"),
    (dict(mass=torch.zeros(2, 3)), "mass must be"),
    (dict(cs=torch.zeros(2, 4)), "cs must be"),
    (dict(angle=torch.zeros(2, 4)), "angle must be"),
    (dict(valid=torch.zeros(2, 4, dtype=torch.bool)), "valid must be"),
    (dict(count=torch.zeros(2, dtype=torch.int64)), "count must be"),
    (dict(count=torch.zeros(3, dtype=torch.int32)), "count must be"),
    (dict(heatmap=torch.zeros(2 * 16 * 24 + 1)[1:].view(2, 1, 16, 24)), None),   # aligned to 4 bytes: accepted up to the device
    (dict(angle=torch.frombuffer(bytearray(68), dtype=torch.float64, offset=4, count=8).view(2, 4)), "angle is misaligned"),
    ({}, "CUDA"),                                   # well-formed CPU tensors: refused for the device, never launched
])
def test_binding_refuses_bad_arguments(over, msg):
    with pytest.raises(cabi.CcvpeError, match=msg or "CUDA"):
        cabi.pose_hypotheses(**_bind_args(**over))


def test_decode_hypotheses_refuses_cpu_tensors():
    with pytest.raises(cabi.CcvpeError, match="CUDA"):
        decode_hypotheses(torch.zeros(1, 1, 8, 8), torch.zeros(1, 2, 8, 8), 2, 1)
    with pytest.raises(cabi.CcvpeError, match="CUDA"):
        models.CVM_VIGOR.decode_hypotheses(torch.zeros(1, 1, 8, 8), torch.zeros(1, 2, 8, 8), 2, 1)


def test_shared_memory_rule():
    lib = cabi.load()
    assert lib.ccvpe_pose_hypotheses_smem_bytes(512, 512) == 143376      # 66 rows of 512 floats + 2 bitmasks of 64 rows
    assert lib.ccvpe_pose_hypotheses_smem_bytes(1, 1) > 0
    assert lib.ccvpe_pose_hypotheses_smem_bytes(64, 1024) > 0
    assert lib.ccvpe_pose_hypotheses_smem_bytes(1024, 1024) == -1        # a 128-row band of 1024 floats is 520 KiB
    assert lib.ccvpe_pose_hypotheses_smem_bytes(0, 512) == -1
    assert lib.ccvpe_pose_hypotheses_smem_bytes(512, -1) == -1


def test_c_abi_refuses_bad_arguments_before_launch():
    """The C entry point checks its arguments itself (the pointers below are never dereferenced)."""
    lib = cabi.load()
    p = ctypes.c_void_p(4096)
    bad = -1                                                                    # CCVPE_ERR_BAD_ARGUMENT

    def call(B=1, H=64, W=64, k=4, radius=2, **ptrs):
        a = dict(heat=p, ori=p, idx=p, rc=p, value=p, mass=p, cs=p, angle=p, valid=p, count=p)
        a.update(ptrs)
        return lib.ccvpe_pose_hypotheses(a["heat"], a["ori"], B, H, W, k, radius, a["idx"], a["rc"], a["value"],
                                         a["mass"], a["cs"], a["angle"], a["valid"], a["count"], None)

    for B, H, W in [(0, 64, 64), (65536, 64, 64), (1, 0, 64), (1, 64, -1)]:
        assert call(B=B, H=H, W=W) == bad and b"bad shape" in lib.ccvpe_last_error(), (B, H, W)
    for k in (0, 65, -1):
        assert call(k=k) == bad and b"k=" in lib.ccvpe_last_error(), k
    for radius in (-1, 32768):
        assert call(radius=radius) == bad and b"radius=" in lib.ccvpe_last_error(), radius
    assert call(H=1024, W=1024) == bad and b"shared memory" in lib.ccvpe_last_error()
    for name in ("heat", "ori", "idx", "rc", "value", "mass", "cs", "angle", "valid", "count"):
        assert call(**{name: None}) == bad and b"null pointer" in lib.ccvpe_last_error(), name
    for name, addr in (("heat", 4097), ("ori", 4098), ("idx", 4100), ("angle", 4100), ("rc", 4098), ("count", 4099)):
        assert call(**{name: ctypes.c_void_p(addr)}) == bad and b"misaligned" in lib.ccvpe_last_error(), name


# ---------------------------------------------------------------------------------------------------------------------
# GPU: exact agreement with the reference
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n_modes,k,radius", [(1, 4, 8), (8, 8, 8), (8, 64, 0), (40, 32, 1), (40, 64, 8), (3, 64, 64)])
def test_mixtures_match_reference(cuda_device, n_modes, k, radius):
    B = 4
    heat = synthetic_mixture(B, n_modes, seed=n_modes * 100 + radius)
    got = check_batch(heat, unit_field(B, 512, 512, seed=n_modes), k, radius, "mixture %d" % n_modes)
    if k >= n_modes and radius == 8:
        assert (got["count"] >= 1).all()


@pytest.mark.gpu
@pytest.mark.parametrize("name,precision", [("vigor_fov360_b2", "fp32"), ("vigor_fov360_b2", "bf16"),
                                            ("kitti_b1", "fp32")])
def test_model_heatmaps_match_reference(cuda_device, name, precision):
    variant, _, noise, circular, _, wseed, _ = GOLDEN_CONFIGS[name]
    model = build_model(variant, noise, circular, wseed).to(cuda_device)
    if precision == "bf16":
        model.set_precision("bf16")
    grd, sat = config_inputs(name)
    with torch.no_grad():
        out = model(grd.to(cuda_device), sat.to(cuda_device))
    heat, ori = out[1].cpu(), out[2].cpu()
    for k, radius in ((8, 4), (32, 16)):
        check_batch(heat, ori, k, radius, "%s %s k=%d r=%d" % (name, precision, k, radius))


def _edge_and_tie_maps():
    """[B, 1, 48, 40]: modes on edges and corners, ties, plateaus, a constant map, +-inf, an all -inf map, NaN maps."""
    H, W = 48, 40
    g = torch.Generator().manual_seed(5)
    base = torch.rand(H, W, generator=g) * 1e-3
    maps = []
    m = base.clone()
    m[0, 0], m[0, W - 1], m[H - 1, 0], m[H - 1, W - 1], m[0, 17], m[H - 1, 3], m[20, 0], m[31, W - 1] = \
        1.0, 0.9, 0.8, 0.7, 0.6, 0.5, 0.4, 0.3
    maps.append(m)
    m = base.clone()
    m[5, 5] = m[5, 30] = m[40, 5] = m[40, 30] = 0.5         # four equal peaks: row-major order
    m[20:23, 10:14] = 0.25                                  # a plateau: every pixel of it is a mode
    maps.append(m)
    maps.append(torch.full((H, W), 0.125))                  # constant: every pixel is a mode
    m = torch.zeros(H, W)
    m[10, 10] = -0.0
    m[3:6, 3:6] = -0.0                                      # -0 and +0 tie
    maps.append(m)
    m = base.clone()
    m[7, 9], m[30, 30], m[12, 25] = INF, INF, -INF          # +-inf as ordinary values; the mass of an inf disc is inf
    maps.append(m)
    maps.append(torch.full((H, W), -INF))                   # all -inf: index 0, like decode_pose
    m = base.clone()
    m[17, 3] = NAN
    maps.append(m)                                          # any NaN: count 0
    maps.append(torch.full((H, W), NAN))
    return torch.stack(maps)[:, None].contiguous()


@pytest.mark.gpu
@pytest.mark.parametrize("k,radius", [(1, 0), (16, 0), (16, 1), (64, 8), (4, 100), (64, 32767)])
def test_edges_ties_plateaus_inf_nan(cuda_device, k, radius):
    heat = _edge_and_tie_maps()
    got = check_batch(heat, unit_field(heat.shape[0], 48, 40, seed=7), k, radius, "edges")
    assert (got["count"][-2:] == 0).all()
    if radius >= 100:                                       # a disc larger than the map claims everything at once
        assert (got["count"][:-2] == 1).all()


@pytest.mark.gpu
@pytest.mark.parametrize("B,H,W,k,radius", [(3, 1, 1, 4, 0), (2, 1, 1000, 64, 2), (2, 1000, 1, 16, 3),
                                            (3, 37, 53, 64, 1), (2, 64, 1024, 32, 8), (5, 9, 7, 64, 0)])
def test_odd_and_small_shapes(cuda_device, B, H, W, k, radius):
    g = torch.Generator().manual_seed(H * 1000 + W)
    heat = torch.rand(B, 1, H, W, generator=g)
    heat[0] = (heat[0] * 8).round() / 8                     # coarse values: ties and plateaus
    check_batch(heat, unit_field(B, H, W, seed=W), k, radius, "%dx%d" % (H, W))


@pytest.mark.gpu
def test_misaligned_heatmap_rows(cuda_device):
    """A heatmap starting 4 bytes past a 16-byte boundary, odd W: each band is loaded through its unaligned ends."""
    B, H, W = 3, 37, 53
    g = torch.Generator().manual_seed(11)
    buf = torch.rand(B * H * W + 1, generator=g).to(cuda_device)
    heat = buf[1:].view(B, 1, H, W)
    ori = unit_field(B, H, W, seed=3).to(cuda_device)
    out = decode_hypotheses(heat, ori, 16, 2)
    got = {key: v.cpu().numpy() for key, v in out.items()}
    h, o = heat.cpu().numpy(), ori.cpu().numpy()
    for b in range(B):
        check_pair(pair(got, b), reference(h[b, 0], o[b], 16, 2), "pair %d" % b)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: buffers, batch independence, graphs
# ---------------------------------------------------------------------------------------------------------------------
OUT_SPECS = (("idx", torch.int64, 1), ("rc", torch.int32, 2), ("value", torch.float32, 1), ("mass", torch.float32, 1),
             ("cs", torch.float32, 2), ("angle", torch.float64, 1), ("valid", torch.uint8, 1), ("count", torch.int32, 0))


def _guarded_outputs(B, k, fill, dev, guard=256):
    """Every output inside its own byte buffer with `guard` bytes of `fill` on each side."""
    bufs, outs = {}, {}
    for name, dt, last in OUT_SPECS:
        shape = (B,) if last == 0 else ((B, k) if last == 1 else (B, k, last))
        nbytes = int(np.prod(shape)) * torch.empty((), dtype=dt).element_size()
        buf = torch.full((guard + nbytes + guard,), fill, dtype=torch.uint8, device=dev)
        bufs[name] = (buf, nbytes)
        outs[name] = buf[guard:guard + nbytes].view(dt).view(shape)
    return bufs, outs


def _launch(heat, ori, k, radius, o):
    cabi.pose_hypotheses(heat, ori, k, radius, o["idx"], o["rc"], o["value"], o["mass"], o["cs"], o["angle"],
                         o["valid"], o["count"])


@pytest.mark.gpu
def test_outputs_written_exactly_once_within_bounds(cuda_device):
    """Two launches into buffers pre-filled with 0x00 and 0xff: the owned bytes agree (every one written, and the result
    is deterministic), the guards keep their fill.  Pairs with count < k cover the empty slots."""
    heat = torch.cat([synthetic_mixture(3, 5, 96, 80, seed=1), torch.full((1, 1, 96, 80), NAN)]).to(cuda_device)
    ori = unit_field(4, 96, 80, seed=2).to(cuda_device)
    k, guard = 64, 256
    runs = []
    for fill in (0x00, 0xFF):
        bufs, outs = _guarded_outputs(4, k, fill, cuda_device, guard)
        _launch(heat, ori, k, 6, outs)
        torch.cuda.synchronize()
        for name, (buf, nbytes) in bufs.items():
            assert bool((buf[:guard] == fill).all()) and bool((buf[guard + nbytes:] == fill).all()), name
        runs.append({name: buf[guard:guard + nbytes].clone() for name, (buf, nbytes) in bufs.items()})
    for name in runs[0]:
        assert torch.equal(runs[0][name], runs[1][name]), name
    count = runs[0]["count"].view(torch.int32).cpu()
    assert count[3] == 0 and (count[:3] < k).all()


@pytest.mark.gpu
def test_batch_permutation_permutes_results(cuda_device):
    B = 6
    heat = synthetic_mixture(B, 12, seed=4).to(cuda_device)
    ori = unit_field(B, 512, 512, seed=4).to(cuda_device)
    perm = torch.tensor([3, 0, 5, 1, 4, 2], device=cuda_device)
    a = decode_hypotheses(heat, ori, 24, 10)
    b = decode_hypotheses(heat[perm], ori[perm], 24, 10)
    for key in KEYS:
        assert torch.equal(a[key][perm].view(torch.uint8), b[key].view(torch.uint8)), key


@pytest.mark.gpu
def test_cuda_graph_replay_with_heatmap_rewritten(cuda_device):
    B, k, radius = 4, 16, 6
    heat = synthetic_mixture(B, 6, seed=8).to(cuda_device)
    ori = unit_field(B, 512, 512, seed=8).to(cuda_device)
    _, outs = _guarded_outputs(B, k, 0, cuda_device)
    _launch(heat, ori, k, radius, outs)                  # warm-up: function attributes are set outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        _launch(heat, ori, k, radius, outs)
    heat.copy_(synthetic_mixture(B, 20, seed=9).to(cuda_device))
    heat[2, 0, 100, 100] = NAN
    graph.replay()
    torch.cuda.synchronize()
    eager = decode_hypotheses(heat, ori, k, radius)
    for key in KEYS:
        assert torch.equal(outs[key].view(torch.uint8), eager[key].view(torch.uint8)), key
    assert int(eager["count"][2]) == 0
