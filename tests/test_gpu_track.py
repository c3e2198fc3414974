"""Sequential location filter (`decoder.track_step`, C ABI `ccvpe_track_step`, `models.track_motion`).

`reference` below is one filter step in NumPy float64: the warp's coordinates in the kernel's operation order (so the taps
and their fractions are the same numbers), the bilinear taps with zero padding and the |det| factor, the two Gaussian
passes with float64 weights, the uniform mix, the product and the normalisation.

Tolerances.  Where every step is exact in float32 (identity or integer-shift motion with sigma = 0, epsilon = 0 or 1) the
device's belief is within 1 float32 ulp of the float64 result rounded once: q is rounded to float32 before it is scaled by
1 / Z, two roundings of which the second can move the result by one ulp.  Z is summed from the float64 products, so the
evidence is within 1e-12.  In general the kernel rounds to float32 at: the 4 bilinear weights, the 4 taps' products and
sums (about 4 u, u = 2^-24), the blur weights (u), each blur pass's accumulations ((2r + 1) u per pass, all terms
non-negative; each tap pair is added before its product: 2 u per d >= 1), q and q / Z (2 u): at most (4r + 9) u =
2.3e-5 relative for r = 96, which the 4e-5 * ref bound covers; the 1e-6 * max(ref) term covers values so small that
float32 subnormals or the float32 weights of a far tail matter.  The evidence sums the same errors over the map, where
they are not all of one sign: 1e-5 relative."""
import ctypes
import math

import numpy as np
import pytest
import torch

from ccvpe_b200 import cabi, models
from ccvpe_b200.decoder import decode_pose, track_step
from ccvpe_b200.models import rotate_matrix, track_motion
from ccvpe_b200.synthetic import GROUND_SHAPES, synthetic_mixture, synthetic_pair, synthetic_track
from helpers import GOLDEN_CONFIGS, build_model

NAN, INF = float("nan"), float("inf")
IDENTITY = [1.0, 0.0, 0.0, 0.0, 1.0, 0.0]


# ---------------------------------------------------------------------------------------------------------------------
# NumPy reference
# ---------------------------------------------------------------------------------------------------------------------
def blur_weights(sigma):
    """w[|d|] for d in [-r, r], float64, normalised; sigma as the C ABI sees it (float32)."""
    sigma = float(np.float32(sigma))
    r = math.ceil(3.0 * sigma)
    if r == 0:
        return np.ones(1)
    w = np.exp(-np.arange(r + 1, dtype=np.float64) ** 2 / (2.0 * sigma * sigma))
    return w / (w[0] + 2.0 * w[1:].sum())


def blur(x, w, axis):
    r = len(w) - 1
    n = x.shape[axis]
    pad = [(0, 0), (0, 0)]
    pad[axis] = (r, r)
    xp = np.pad(x, pad)
    out = np.zeros_like(x)
    for d in range(-r, r + 1):
        sl = [slice(None), slice(None)]
        sl[axis] = slice(r + d, r + d + n)
        out += w[abs(d)] * xp[tuple(sl)]
    return out


def warp(b, a):
    """The old belief b [H, W] on the new grid: bilinear at (v, u), zero padding, times |det|."""
    H, W = b.shape
    a0, a1, a2, a3, a4, a5 = [float(v) for v in a]
    jj, ii = np.meshgrid(np.arange(W, dtype=np.float64), np.arange(H, dtype=np.float64))
    xc, yc = jj + 0.5, ii + 0.5
    with np.errstate(invalid="ignore", over="ignore"):
        u = ((a0 * xc + a1 * yc) + a2) - 0.5
        v = ((a3 * xc + a4 * yc) + a5) - 0.5
        uf, vf = np.floor(u), np.floor(v)
        inside = (uf >= -1) & (uf <= W - 1) & (vf >= -1) & (vf <= H - 1)
        dx, dy = np.where(inside, u - uf, 0.0), np.where(inside, v - vf, 0.0)
    x0, y0 = np.where(inside, uf, 0).astype(np.int64), np.where(inside, vf, 0).astype(np.int64)
    b64 = b.astype(np.float64)
    p = np.zeros((H, W))
    with np.errstate(invalid="ignore"):
        for oy, wy in ((0, 1.0 - dy), (1, dy)):
            for ox, wx in ((0, 1.0 - dx), (1, dx)):
                y, x = y0 + oy, x0 + ox
                ok = inside & (y >= 0) & (y < H) & (x >= 0) & (x < W)
                p += np.where(ok, wy * wx * b64[np.clip(y, 0, H - 1), np.clip(x, 0, W - 1)], 0.0)
        det = abs(a0 * a4 - a1 * a3)
        return np.where(inside, p * det, 0.0)


def reference(belief, heat, a, sigma, eps):
    """One track: belief, heat float32 [H, W]; a: 6 floats.  Returns (new belief float64, evidence, reset)."""
    H, W = heat.shape
    eps = float(np.float32(eps))
    w = blur_weights(sigma)
    with np.errstate(invalid="ignore", over="ignore"):
        p = blur(blur(warp(belief, a), w, 1), w, 0)
        prior = (1.0 - eps) * p + eps / (H * W)
        q = prior * heat.astype(np.float64)
        z = q.sum()
    if z > 0 and math.isfinite(z):
        return q / z, z, 0
    return heat.astype(np.float64), z, 1


def run(belief, heat, motion, sigma, eps):
    """Device step on copies; returns (belief, evidence, reset) as NumPy arrays."""
    dev = torch.device("cuda:0")
    bel = belief.clone().to(dev)
    out = track_step(bel, heat.to(dev), torch.as_tensor(motion, dtype=torch.float64).to(dev), sigma, eps)
    torch.cuda.synchronize()
    return bel.cpu().numpy(), out["evidence"].cpu().numpy(), out["reset"].cpu().numpy()


def check_general(belief, heat, motion, sigma, eps, where=""):
    got, ev, rs = run(belief, heat, motion, sigma, eps)
    motion = np.asarray(motion, np.float64).reshape(-1, 6)
    for b in range(heat.shape[0]):
        ref, z, reset = reference(belief[b, 0].numpy(), heat[b, 0].numpy(), motion[b], sigma, eps)
        assert rs[b] == reset, (where, b, z)
        if reset:
            assert np.array_equal(got[b, 0].view(np.uint32), heat[b, 0].numpy().view(np.uint32)), (where, b)
            continue
        err = np.abs(got[b, 0].astype(np.float64) - ref)
        bound = 4e-5 * ref + 1e-6 * ref.max()
        assert (err <= bound).all(), (where, b, float((err / np.maximum(bound, 1e-300)).max()))
        assert abs(ev[b] - z) <= 1e-5 * z, (where, b, ev[b], z)
    return got, ev, rs


def check_tight(belief, heat, motion, sigma, eps, where=""):
    """belief within 1 float32 ulp of the float64 result rounded once, evidence within 1e-12.  Where q itself is below
    float32's normal range its rounding to float32 is absolute (at most half the subnormal spacing, 2^-150), which the
    division by Z scales to 2^-150 / Z."""
    got, ev, rs = run(belief, heat, motion, sigma, eps)
    motion = np.asarray(motion, np.float64).reshape(-1, 6)
    for b in range(heat.shape[0]):
        ref, z, reset = reference(belief[b, 0].numpy(), heat[b, 0].numpy(), motion[b], sigma, eps)
        assert rs[b] == 0 and reset == 0, (where, b)
        ref32 = ref.astype(np.float32)
        ulp = np.spacing(np.abs(ref32)).astype(np.float64)
        ulp = np.where(ref * z < 2.0 ** -126, ulp + 2.0 ** -150 / z, ulp)
        assert (np.abs(got[b, 0].astype(np.float64) - ref32) <= ulp).all(), (where, b)
        assert abs(ev[b] - z) <= 1e-12 * z, (where, b, ev[b], z)
    return got, ev


def mixture(B, H, W, seed, n_modes=6, floor=0.0):
    """synthetic_mixture maps; far from every mode they underflow to 0, so a heatmap gets a floor where a step must not
    reset on disjoint supports."""
    return synthetic_mixture(B, n_modes, H, W, seed=seed) + floor


def crop(left, top, angle=0.0, scale=1.0, size=(512, 512)):
    """Affine data of a crop cut from a map: rotated by `angle` about its centre, scaled, at (left, top)."""
    m = rotate_matrix(angle, size) if angle else list(IDENTITY)
    m = [m[0] * scale, m[1] * scale, m[2] * scale, m[3] * scale, m[4] * scale, m[5] * scale]
    m[2] += left
    m[5] += top
    return m


# ---------------------------------------------------------------------------------------------------------------------
# CPU: track_motion, the reference, every refusal
# ---------------------------------------------------------------------------------------------------------------------
def test_track_motion_hand_worked():
    # a crop at twice the map's scale: the map offset (4, 8) is (2, 4) crop pixels
    assert track_motion([2, 0, 10, 0, 2, 20], [2, 0, 14, 0, 2, 28]) == [1.0, 0.0, 2.0, 0.0, 1.0, 4.0]
    # the vehicle moved by (2, 4) map pixels: the new position came from (14 - 2 - 10, 28 - 4 - 20) / 2
    assert track_motion([2, 0, 10, 0, 2, 20], [2, 0, 14, 0, 2, 28], (2, 4)) == [1.0, 0.0, 1.0, 0.0, 1.0, 2.0]
    # previous crop turned a quarter: its inverse is [0 1; -1 0], applied to the new crop's offset (3, 5)
    m = track_motion([0, -1, 0, 1, 0, 0], [1, 0, 3, 0, 1, 5])
    assert m == [0.0, 1.0, 5.0, -1.0, 0.0, -3.0]


def test_track_motion_translation_is_exact():
    for left0, top0, left1, top1, sx, sy in [(100, 37, 104, 30, 3.25, -6.75), (0, 0, -3, 9, 0.1, 0.7),
                                             (2048, 4096, 2051, 4093, 2.9, -3.3)]:
        m = track_motion([1, 0, left0, 0, 1, top0], [1, 0, left1, 0, 1, top1], (sx, sy))
        assert m == [1.0, 0.0, (left1 - sx) - left0, 0.0, 1.0, (top1 - sy) - top0]


def test_track_motion_round_trips_with_rotate_matrix():
    """A_prev(M(q)) + shift == A_new(q) for rotated, scaled and shifted crops; equal crops give the identity."""
    rng = np.random.default_rng(0)
    for angle0, angle1, s0, s1 in [(0, 10, 1, 1), (33.3, -20, 1, 1.2), (190, 185, 0.8, 0.8), (90, 270, 1, 1)]:
        prev, new = crop(500, 700, angle0, s0), crop(512.5, 690, angle1, s1)
        shift = (4.5, -7.25)
        m = track_motion(prev, new, shift)
        for x, y in rng.uniform(0, 512, (8, 2)):
            mx, my = m[0] * x + m[1] * y + m[2], m[3] * x + m[4] * y + m[5]
            px, py = prev[0] * mx + prev[1] * my + prev[2], prev[3] * mx + prev[4] * my + prev[5]
            nx, ny = new[0] * x + new[1] * y + new[2], new[3] * x + new[4] * y + new[5]
            assert abs(px + shift[0] - nx) < 1e-9 and abs(py + shift[1] - ny) < 1e-9
        np.testing.assert_allclose(track_motion(new, new), IDENTITY, atol=1e-12)
    with pytest.raises(ValueError, match="not invertible"):
        track_motion([1, 2, 0, 2, 4, 0], IDENTITY)


def test_reference_hand_worked():
    """Identity motion, sigma 0: the belief times the heatmap, normalised; a shift of one column right moves the belief
    (its first column leaves the crop); epsilon 1 gives the normalised heatmap; disjoint supports reset."""
    b = np.array([[0.5, 0.25, 0.25]], np.float32)
    h = np.array([[0.2, 0.2, 0.6]], np.float32)
    ref, z, reset = reference(b, h, IDENTITY, 0, 0)
    assert reset == 0 and abs(z - 0.3) < 1e-7
    np.testing.assert_allclose(ref, [[1 / 3, 1 / 6, 1 / 2]], rtol=1e-7)
    ref, z, _ = reference(b, h, [1, 0, -1, 0, 1, 0], 0, 0)        # new column j came from old column j - 1
    np.testing.assert_allclose(ref, [[0, 0.4, 0.6]], rtol=1e-7)                  # p = [0, 0.5, 0.25], Z = 0.25
    ref, z, _ = reference(b, h, IDENTITY, 0, 1)
    np.testing.assert_allclose(ref, h / h.sum(), rtol=1e-7)
    ref, z, reset = reference(np.array([[1, 0, 0]], np.float32), np.array([[0, 1, 0]], np.float32), IDENTITY, 0, 0)
    assert reset == 1 and z == 0
    # a half-pixel shift averages neighbours; scale 2 doubles the density it samples (|det| = 4 for a 2x zoom out)
    ref = warp(np.array([[0.0, 1.0, 0.0, 0.0]], np.float32), [1, 0, 0.5, 0, 1, 0])
    np.testing.assert_allclose(ref, [[0.5, 0.5, 0.0, 0.0]])
    assert warp(np.ones((4, 4), np.float32), [2, 0, 0, 0, 2, 0])[0, 0] == 4.0
    w = blur_weights(2.0)
    assert len(w) == 7 and abs(w[0] + 2 * w[1:].sum() - 1) < 1e-15


def _bind(B=2, H=16, W=24, **over):
    a = dict(belief=torch.zeros(B, 1, H, W), heatmap=torch.zeros(B, 1, H, W), motion=torch.zeros(B, 6, dtype=torch.float64),
             sigma=2.0, epsilon=0.0, evidence=torch.zeros(B, dtype=torch.float64), reset=torch.zeros(B, dtype=torch.uint8),
             scratch=torch.zeros(max(cabi.track_scratch_bytes(B, H, W), 8), dtype=torch.uint8))
    a.update(over)
    return a


_shared = torch.zeros(2 * 2 * 16 * 24 + 8)


@pytest.mark.parametrize("over,msg", [
    (dict(sigma=-0.5), "sigma must be"), (dict(sigma=32.5), "sigma must be"), (dict(sigma=NAN), "sigma must be"),
    (dict(sigma=INF), "sigma must be"), (dict(sigma=True), "sigma must be"), (dict(sigma="2"), "sigma must be"),
    (dict(epsilon=-1e-9), "epsilon must be"), (dict(epsilon=1.5), "epsilon must be"), (dict(epsilon=NAN), "epsilon must be"),
    (dict(belief=torch.zeros(2, 1, 16, 24, dtype=torch.float64)), "belief must be a float32"),
    (dict(belief=torch.zeros(2, 16, 24)), "belief must have shape"),
    (dict(belief=torch.zeros(2, 1, 24, 16).transpose(2, 3)), "belief must be contiguous"),
    (dict(belief=torch.zeros(0, 1, 16, 24)), "1 <= B"),
    (dict(belief=torch.zeros(1, 1, 4097, 1), heatmap=torch.zeros(1, 1, 4097, 1)), "H, W <= 4096"),
    (dict(heatmap=torch.zeros(2, 1, 16, 25)), "heatmap must have shape"),
    (dict(heatmap=torch.zeros(2, 1, 16, 24, dtype=torch.bfloat16)), "heatmap must be a float32"),
    (dict(motion=torch.zeros(2, 6)), "motion must be"), (dict(motion=torch.zeros(2, 5, dtype=torch.float64)), "motion must be"),
    (dict(motion=torch.zeros(6, 2, dtype=torch.float64).t()), "motion must be"),
    (dict(evidence=torch.zeros(2)), "evidence must be"), (dict(evidence=torch.zeros(3, dtype=torch.float64)), "evidence must be"),
    (dict(reset=torch.zeros(2, dtype=torch.bool)), "reset must be"),
    (dict(scratch=torch.zeros(16, dtype=torch.uint8)), "scratch must be"),
    (dict(scratch=torch.zeros(1 << 20)), "scratch must be"),
    (dict(motion=torch.frombuffer(bytearray(100), dtype=torch.float64, offset=4, count=12).view(2, 6)), "motion is misaligned"),
    (dict(belief=_shared[:768].view(2, 1, 16, 24), heatmap=_shared[8:776].view(2, 1, 16, 24)), "overlaps"),
    (dict(heatmap="belief"), "overlaps"),
    ({}, "CUDA"),                                   # well-formed CPU tensors: refused for the device, never launched
])
def test_binding_refuses_bad_arguments(over, msg):
    a = _bind(**over)
    if isinstance(a["heatmap"], str):
        a["heatmap"] = a["belief"]
    with pytest.raises(cabi.CcvpeError, match=msg):
        cabi.track_step(**a)


def test_track_step_refuses_cpu_tensors():
    for fn in (track_step, models.CVM_OxfordRobotCar.track_step):
        with pytest.raises(cabi.CcvpeError, match="CUDA"):
            fn(torch.zeros(1, 1, 8, 8), torch.zeros(1, 1, 8, 8), torch.zeros(1, 6, dtype=torch.float64), 1.0)


def test_scratch_rule():
    lib = cabi.load()
    # 16 x 8 tiles of 32 x 64 -> 128 float64 partials (1 KiB, rounded to 256 B), then the 512 x 512 float32 plane
    assert lib.ccvpe_track_scratch_bytes(1, 512, 512) == 1024 + 512 * 512 * 4
    assert lib.ccvpe_track_scratch_bytes(64, 512, 512) == 64 * 1024 + 64 * 512 * 512 * 4
    assert lib.ccvpe_track_scratch_bytes(1, 1, 1) == 256 + 4
    for B, H, W in [(0, 8, 8), (65536, 8, 8), (1, 0, 8), (1, 8, 4097), (1, -1, 8)]:
        assert lib.ccvpe_track_scratch_bytes(B, H, W) == -1, (B, H, W)


def test_c_abi_refuses_bad_arguments_before_launch():
    """The C entry point checks its arguments itself (the pointers below are never dereferenced)."""
    lib = cabi.load()
    bad = -1                                                                    # CCVPE_ERR_BAD_ARGUMENT

    def call(B=1, H=64, W=64, sigma=1.0, eps=0.0, **ptrs):
        a = dict(belief=1 << 20, heat=1 << 30, motion=4096, evidence=8192, reset=12288, scratch=1 << 32)
        a.update(ptrs)
        a = {k: ctypes.c_void_p(v) for k, v in a.items()}
        return lib.ccvpe_track_step(a["belief"], a["heat"], a["motion"], B, H, W, sigma, eps, a["evidence"], a["reset"],
                                    a["scratch"], None)

    for B, H, W in [(0, 64, 64), (65536, 64, 64), (1, 0, 64), (1, 64, -1), (1, 4097, 8), (1, 8, 4097)]:
        assert call(B=B, H=H, W=W) == bad and b"bad shape" in lib.ccvpe_last_error(), (B, H, W)
    for sigma in (-1.0, 32.5, NAN, INF):
        assert call(sigma=sigma) == bad and b"sigma=" in lib.ccvpe_last_error(), sigma
    for eps in (-0.1, 1.5, NAN):
        assert call(eps=eps) == bad and b"epsilon=" in lib.ccvpe_last_error(), eps
    for name in ("belief", "heat", "motion", "evidence", "reset", "scratch"):
        assert call(**{name: 0}) == bad and b"null pointer" in lib.ccvpe_last_error(), name
    for name, addr in (("belief", (1 << 20) + 2), ("heat", (1 << 30) + 1), ("motion", 4100), ("evidence", 8196),
                       ("scratch", (1 << 32) + 4)):
        assert call(**{name: addr}) == bad and b"misaligned" in lib.ccvpe_last_error(), name
    assert call(heat=(1 << 20) + 64 * 64 * 4 - 4) == bad and b"overlaps" in lib.ccvpe_last_error()
    assert call(heat=(1 << 20) - 64 * 64 * 4 + 4) == bad and b"overlaps" in lib.ccvpe_last_error()


def test_synthetic_track_is_seeded_and_consistent():
    a, b = synthetic_track(6, 2, 128, 96, seed=3), synthetic_track(6, 2, 128, 96, seed=3)
    for key in a:
        assert torch.equal(a[key], b[key]), key
    assert a["heatmap"].shape == (6, 2, 1, 128, 96) and a["motion"].dtype == torch.float64
    assert torch.equal(a["motion"][0], torch.tensor([IDENTITY] * 2, dtype=torch.float64))
    # the true motion maps each frame's true position onto the previous frame's (pixel centres: index + 0.5)
    for t in range(1, 6):
        for k in range(2):
            m = a["motion"][t, k].tolist()
            y, x = (a["truth"][t, k] + 0.5).tolist()
            py, px = (a["truth"][t - 1, k] + 0.5).tolist()
            assert abs(m[0] * x + m[1] * y + m[2] - px) < 1e-9 and abs(m[3] * x + m[4] * y + m[5] - py) < 1e-9


# ---------------------------------------------------------------------------------------------------------------------
# GPU: tight cases
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("H,W", [(512, 512), (37, 53), (1, 1)])
def test_identity_motion_is_the_normalised_product(cuda_device, H, W):
    B = 3
    bel, heat = mixture(B, H, W, seed=1), mixture(B, H, W, seed=2, floor=1e-7)
    check_tight(bel, heat, [IDENTITY] * B, 0.0, 0.0, "identity %dx%d" % (H, W))


@pytest.mark.gpu
def test_integer_translations(cuda_device):
    """sigma = 0, shifts of whole pixels: the belief moves without interpolation, the mass that leaves the crop is lost."""
    shifts = [(0, 0), (1, 0), (0, -1), (-17, 23), (200, -311), (-511, 511)]
    B = len(shifts)
    bel = mixture(B, 512, 512, seed=3, n_modes=12, floor=1e-7)     # the last shift keeps one pixel of it
    heat = mixture(B, 512, 512, seed=4, n_modes=12, floor=1e-7)
    motion = [[1, 0, float(dx), 0, 1, float(dy)] for dx, dy in shifts]
    check_tight(bel, heat, motion, 0.0, 0.0, "integer shifts")
    check_tight(bel, heat, motion, 0.0, 1.0, "integer shifts, epsilon 1")


@pytest.mark.gpu
@pytest.mark.parametrize("H,W", [(512, 512), (31, 17)])
def test_epsilon_one_gives_the_normalised_heatmap(cuda_device, H, W):
    B = 2
    bel, heat = mixture(B, H, W, seed=5), mixture(B, H, W, seed=6, floor=1e-7)
    got, ev = check_tight(bel, heat, [crop(3.3, -2.1, 17.0)] * B, 8.0, 1.0, "epsilon 1")
    h = heat.double().numpy()
    ref = (h / h.sum(axis=(2, 3), keepdims=True)).astype(np.float32)
    assert (np.abs(got.astype(np.float64) - ref) <= np.spacing(np.abs(ref))).all()


# ---------------------------------------------------------------------------------------------------------------------
# GPU: general cases
# ---------------------------------------------------------------------------------------------------------------------
def _motions(B, size=(512, 512)):
    """rotation about the centre + sub-pixel shift, a 1.1x zoom, a translation, the identity, ..."""
    W, H = size
    out = [track_motion(crop(1000, 2000, 10.0, size=size), crop(1003.3, 1994.6, 14.5, size=size), (0.25, -1.75)),
           track_motion(crop(1000, 2000, 0.0, 1.0, size), crop(990, 1990, 0.0, 1.1, size), (0.0, 0.0)),
           [1.0, 0.0, 2.4, 0.0, 1.0, -0.7], IDENTITY,
           track_motion(crop(0, 0, 200.0, 0.9, size), crop(5, 5, 170.0, 1.0, size), (-W / 8, H / 16))]
    return [out[k % len(out)] for k in range(B)]


@pytest.mark.gpu
@pytest.mark.parametrize("sigma", [0.0, 0.5, 2.0, 8.0, 32.0])
@pytest.mark.parametrize("eps", [0.0, 1e-3, 0.5, 1.0])
def test_mixtures_match_reference(cuda_device, sigma, eps):
    B = 5
    bel = mixture(B, 512, 512, seed=int(sigma * 10) + 7, n_modes=8)
    heat = mixture(B, 512, 512, seed=int(eps * 1000) + 8, n_modes=8, floor=1e-7)
    _, _, rs = check_general(bel, heat, _motions(B), sigma, eps, "sigma %g eps %g" % (sigma, eps))
    assert not rs.any()


@pytest.mark.gpu
@pytest.mark.parametrize("name,shape_key", [("oxford_b1", "oxford"), ("vigor_fov360_b2", "vigor")])
def test_model_heatmaps_match_reference(cuda_device, name, shape_key):
    """bf16 model heatmaps of two frames: the first is the belief, the second the heatmap of the step."""
    variant, _, noise, circular, _, wseed, _ = GOLDEN_CONFIGS[name]
    model = build_model(variant, noise, circular, wseed).to(cuda_device)
    model.set_precision("bf16")
    frames = []
    for seed in (11, 12):
        grd, sat = synthetic_pair(2, GROUND_SHAPES[shape_key], seed=seed)
        with torch.no_grad():
            frames.append(model(grd.to(cuda_device), sat.to(cuda_device))[1].cpu())
    for sigma, eps in ((2.0, 1e-3), (8.0, 0.0), (0.5, 0.5)):
        check_general(frames[0], frames[1], _motions(2), sigma, eps, "%s sigma %g eps %g" % (name, sigma, eps))


@pytest.mark.gpu
@pytest.mark.parametrize("B,H,W", [(3, 1, 1), (2, 1, 7), (2, 5, 1), (2, 37, 53), (2, 3, 300), (2, 300, 3), (1, 129, 65)])
@pytest.mark.parametrize("sigma", [0.0, 2.0, 32.0])
def test_odd_and_small_shapes(cuda_device, B, H, W, sigma):
    g = torch.Generator().manual_seed(H * 1000 + W)
    bel, heat = torch.rand(B, 1, H, W, generator=g), torch.rand(B, 1, H, W, generator=g)
    motion = _motions(B, (W, H))
    if H * W == 1:
        motion = [IDENTITY, [1, 0, 0.25, 0, 1, -0.5], [0.5, 0, 0, 0, 0.5, 0]][:B]
    check_general(bel, heat, motion, sigma, 1e-3, "%dx%d" % (H, W))


# ---------------------------------------------------------------------------------------------------------------------
# GPU: edge cases
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_resets_copy_the_heatmap(cuda_device):
    """Disjoint support with epsilon 0, a NaN, a +inf and an all-zero heatmap: reset, and the heatmap's bits."""
    H = W = 64
    bel = torch.zeros(5, 1, H, W)
    bel[:, :, :, :32] = 1.0 / (H * 32)
    heat = mixture(5, H, W, seed=9, floor=1e-7)
    heat[0, :, :, :40] = 0.0                                   # disjoint after a shift of 8 columns to the right
    heat[1, 0, 10, 10] = NAN
    heat[2, 0, 20, 5] = INF
    heat[3] = 0.0
    motion = [[1, 0, -8, 0, 1, 0]] + [IDENTITY] * 4
    got, ev, rs = check_general(bel, heat, motion, 0.0, 0.0, "resets")
    assert rs.tolist() == [1, 1, 1, 1, 0]
    assert ev[0] == 0 and math.isnan(ev[1]) and ev[2] == INF and ev[3] == 0
    assert np.array_equal(got[:4].view(np.uint32), heat[:4].numpy().view(np.uint32))


@pytest.mark.gpu
def test_nan_belief_recovers_on_the_next_finite_frame(cuda_device):
    dev = cuda_device
    bel = mixture(2, 96, 80, seed=10).to(dev)
    bel[0, 0, 40, 40] = NAN
    heats = [mixture(2, 96, 80, seed=s, floor=1e-7).to(dev) for s in (11, 12)]
    motion = torch.tensor([[1, 0, 0.5, 0, 1, -0.25]] * 2, dtype=torch.float64, device=dev)
    r1 = track_step(bel, heats[0], motion, 2.0, 1e-3)
    assert r1["reset"].tolist() == [1, 0] and math.isnan(float(r1["evidence"][0]))
    assert torch.equal(bel[0], heats[0][0])
    before = bel.cpu()
    r2 = track_step(bel, heats[1], motion, 2.0, 1e-3)
    assert r2["reset"].tolist() == [0, 0] and bool(torch.isfinite(bel).all())
    for b in range(2):
        ref, z, _ = reference(before[b, 0].numpy(), heats[1][b, 0].cpu().numpy(), motion[b].tolist(), 2.0, 1e-3)
        err = np.abs(bel[b, 0].cpu().numpy().astype(np.float64) - ref)
        assert (err <= 4e-5 * ref + 1e-6 * ref.max()).all()


@pytest.mark.gpu
@pytest.mark.parametrize("eps", [0.0, 0.25])
def test_non_finite_and_huge_motion(cuda_device, eps):
    """A NaN, inf or 1e12-pixel motion predicts nothing inside the crop: with epsilon 0 the track resets, otherwise the
    prior is uniform and the belief is the normalised heatmap."""
    motions = [[NAN, 0, 0, 0, 1, 0], [1, 0, NAN, 0, 1, 0], [1, 0, INF, 0, 1, 0], [1, 0, 0, 0, 1, -INF],
               [INF, 0, 0, 0, INF, 0], [1, 0, 1e12, 0, 1, 0], [1, 0, 0, 0, 1, -1e12], [1e12, 0, 0, 0, 1e12, 0]]
    B = len(motions)
    bel, heat = mixture(B, 64, 64, seed=13), mixture(B, 64, 64, seed=14, floor=1e-7)
    got, ev, rs = check_general(bel, heat, motions, 2.0, eps, "motion eps %g" % eps)
    assert (rs == (1 if eps == 0 else 0)).all()


@pytest.mark.gpu
def test_guarded_outputs_and_in_place_equals_a_copy(cuda_device):
    """belief, evidence and reset inside buffers with 256 guard bytes of 0x00 / 0xff on each side: the guards keep their
    fill, and the result equals the same step on a plain contiguous copy of the belief."""
    dev, B, H, W, guard = cuda_device, 4, 100, 130, 256
    bel0 = mixture(B, H, W, seed=15).to(dev)
    heat = mixture(B, H, W, seed=16, floor=1e-7).to(dev)
    heat[3] = 0.0                                              # one reset
    motion = torch.tensor(_motions(B, (W, H)), dtype=torch.float64, device=dev)
    plain = bel0.clone()
    ref = track_step(plain, heat, motion, 3.0, 1e-2)
    for fill in (0x00, 0xFF):
        bufs = {}
        for name, nbytes in (("belief", B * H * W * 4), ("evidence", B * 8), ("reset", B)):
            bufs[name] = (torch.full((guard + nbytes + guard,), fill, dtype=torch.uint8, device=dev), nbytes)
        bel = bufs["belief"][0][guard:guard + B * H * W * 4].view(torch.float32).view(B, 1, H, W)
        bel.copy_(bel0)
        ev = bufs["evidence"][0][guard:guard + B * 8].view(torch.float64)
        rs = bufs["reset"][0][guard:guard + B]
        scratch = torch.full((cabi.track_scratch_bytes(B, H, W),), fill, dtype=torch.uint8, device=dev)
        cabi.track_step(bel, heat, motion, 3.0, 1e-2, ev, rs, scratch)
        torch.cuda.synchronize()
        for name, (buf, nbytes) in bufs.items():
            assert bool((buf[:guard] == fill).all()) and bool((buf[guard + nbytes:] == fill).all()), name
        assert torch.equal(bel.view(torch.int32), plain.view(torch.int32))
        assert torch.equal(ev.view(torch.int64), ref["evidence"].view(torch.int64))
        assert torch.equal(rs, ref["reset"]) and rs.tolist() == [0, 0, 0, 1]


@pytest.mark.gpu
def test_batch_permutation_permutes_results(cuda_device):
    dev, B = cuda_device, 6
    bel = mixture(B, 512, 512, seed=17).to(dev)
    heat = mixture(B, 512, 512, seed=18, floor=1e-7).to(dev)
    motion = torch.tensor(_motions(B), dtype=torch.float64, device=dev)
    perm = torch.tensor([3, 0, 5, 1, 4, 2], device=dev)
    a, b = bel.clone(), bel[perm].contiguous()
    ra = track_step(a, heat, motion, 8.0, 1e-3)
    rb = track_step(b, heat[perm].contiguous(), motion[perm].contiguous(), 8.0, 1e-3)
    assert torch.equal(a[perm].view(torch.int32), b.view(torch.int32))
    assert torch.equal(ra["evidence"][perm].view(torch.int64), rb["evidence"].view(torch.int64))
    assert torch.equal(ra["reset"][perm], rb["reset"])


# ---------------------------------------------------------------------------------------------------------------------
# GPU: determinism, graphs, behaviour
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_two_eager_runs_are_equal(cuda_device):
    dev, B = cuda_device, 8
    bel = mixture(B, 512, 512, seed=19).to(dev)
    heat = mixture(B, 512, 512, seed=20, floor=1e-7).to(dev)
    motion = torch.tensor(_motions(B), dtype=torch.float64, device=dev)
    outs = []
    for _ in range(2):
        b = bel.clone()
        r = track_step(b, heat, motion, 32.0, 1e-3)
        outs.append((b, r["evidence"], r["reset"]))
    for x, y in zip(*outs):
        assert torch.equal(x, y)


@pytest.mark.gpu
def test_cuda_graph_sequence_equals_eager(cuda_device):
    """One step captured once, replayed for 19 frames with the heatmap and motion rewritten in place before each replay."""
    dev, T, B = cuda_device, 20, 3
    seq = synthetic_track(T, B, 256, 320, seed=1)
    heats, motions = seq["heatmap"].to(dev), seq["motion"].to(dev)
    eager = heats[0].clone()
    eager_out = []
    for t in range(1, T):
        r = track_step(eager, heats[t], motions[t], 1.5, 1e-3)
        eager_out.append((eager.clone(), r["evidence"].clone(), r["reset"].clone()))
    bel, heat, motion = heats[0].clone(), torch.empty_like(heats[0]), torch.empty_like(motions[0])
    ev, rs = torch.empty(B, dtype=torch.float64, device=dev), torch.empty(B, dtype=torch.uint8, device=dev)
    scratch = torch.empty(cabi.track_scratch_bytes(B, 256, 320), dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        cabi.track_step(bel, heat, motion, 1.5, 1e-3, ev, rs, scratch)
    for t in range(1, T):
        heat.copy_(heats[t])
        motion.copy_(motions[t])
        graph.replay()
        b, e, r = eager_out[t - 1]
        assert torch.equal(bel, b) and torch.equal(ev, e) and torch.equal(rs, r), t
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_filter_follows_the_trajectory_through_distractors(cuda_device):
    """On synthetic_track, the filtered belief's argmax stays within 3 pixels of the true position on every frame, while
    the frame's own argmax jumps to the stronger distractor on the frames where it is stronger."""
    dev, T, B = cuda_device, 30, 2
    seq = synthetic_track(T, B, seed=0)
    heats, motions = seq["heatmap"].to(dev), seq["motion"].to(dev)
    ori = torch.zeros(B, 2, 512, 512, device=dev)
    bel = heats[0].clone()
    assert int(seq["strong"].sum()) >= 6
    for t in range(1, T):
        r = track_step(bel, heats[t], motions[t], 1.5, 1e-3)
        assert not r["reset"].any() and bool((r["evidence"] > 0).all()), t
        fused = decode_pose(bel, ori)["rc"].cpu().double()
        raw = decode_pose(heats[t], ori)["rc"].cpu().double()
        assert ((fused - seq["truth"][t]).norm(dim=1) <= 3.0).all(), (t, fused, seq["truth"][t])
        for b in range(B):
            target = seq["distractor"][t, b] if seq["strong"][t, b] else seq["truth"][t, b]
            assert float((raw[b] - target).norm()) <= 3.0, (t, b, raw[b], target)
