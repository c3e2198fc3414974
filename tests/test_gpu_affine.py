"""Device bilinear affine transform / rotation (ccvpe_affine_u8, `model.affine_u8` / `model.rotate_u8`) against its oracle,
Pillow itself: Image.transform(size, AFFINE, data, BILINEAR, fillcolor) and Image.rotate(angle, BILINEAR, center, translate,
fillcolor).  Every comparison is exact (torch.equal)."""
import ctypes
import functools
import itertools
import math

import numpy as np
import pytest
import torch
from PIL import Image

from ccvpe_b200 import cabi, models
from ccvpe_b200.models import rotate_matrix
from helpers import OUT_NAMES, build_model

affine_u8 = models.CVM_VIGOR.affine_u8
rotate_u8 = models.CVM_VIGOR.rotate_u8
B = 3
CONTENTS = ["noise", "gradient", "saturated"]


def _rot(deg, W, H, s=1.0, cx=None, cy=None, tx=0.0, ty=0.0):
    """output -> input matrix of a rotation by `deg` (scaled by 1 / s) about (cx, cy), then shifted by (tx, ty)"""
    cx, cy = (W / 2 if cx is None else cx), (H / 2 if cy is None else cy)
    c, n = math.cos(math.radians(deg)) / s, math.sin(math.radians(deg)) / s
    return [c, n, cx - c * (cx + tx) - n * (cy + ty), -n, c, cy + n * (cx + tx) - c * (cy + ty)]


#: name -> ((H, W), (h, w), (left, top), three matrices (one per image), fill).  Rotations by +-10 degrees and arbitrary
#: angles, quarter turns and 180 on square and non-square images, flips, integer and fractional shifts, 0.3x-3x scales,
#: shear, a matrix that maps every pixel outside (all fill), 1x1 and 1xN images, outputs larger and smaller than the
#: input, and the 1280x1280 -> 512x512 rotate + centre crop
CASES = {
    "rot10": ((97, 131), (97, 131), (0, 0), [_rot(10, 131, 97), _rot(-10, 131, 97), _rot(9.75, 131, 97, tx=3, ty=-2)],
              (0, 0, 0)),
    "rot_any": ((192, 256), (192, 256), (0, 0), [_rot(37.3, 256, 192), _rot(-123.7, 256, 192, cx=10.5, cy=170.25),
                                                 _rot(200.1, 256, 192)], (12, 200, 255)),
    "quarter_square": ((64, 64), (64, 64), (0, 0), [rotate_matrix(a, (64, 64)) for a in (90, 180, 270)], (0, 0, 0)),
    "quarter_rect": ((45, 80), (45, 80), (0, 0), [rotate_matrix(a, (80, 45)) for a in (90, 180, 270)], (7, 8, 9)),
    "flips": ((50, 70), (50, 70), (0, 0), [[-1.0, 0.0, 70.0, 0.0, 1.0, 0.0], [1.0, 0.0, 0.0, 0.0, -1.0, 50.0],
                                           [0.0, 1.0, 0.0, 1.0, 0.0, 0.0]], (0, 0, 0)),
    "shifts": ((60, 90), (60, 90), (0, 0), [[1.0, 0.0, 5.0, 0.0, 1.0, -3.0], [1.0, 0.0, 0.25, 0.0, 1.0, -7.6],
                                            [1.0, 0.0, -0.3333, 0.0, 1.0, 0.5]], (255, 0, 128)),
    "scales": ((120, 100), (120, 100), (0, 0), [_rot(0, 100, 120, s=0.3), _rot(0, 100, 120, s=3.0),
                                                [1.7, 0.0, -20.0, 0.0, 0.45, 13.0]], (0, 0, 0)),
    "shear": ((80, 80), (80, 80), (0, 0), [[1.0, 0.3, -5.0, 0.2, 1.0, 0.0], [1.0, -0.45, 12.0, 0.0, 1.0, 0.0],
                                           _rot(25, 80, 80, s=1.3)], (0, 0, 0)),
    "all_outside": ((33, 47), (20, 30), (0, 0), [[1.0, 0.0, 1e4, 0.0, 1.0, 0.0], [1.0, 0.0, 0.0, 0.0, 1.0, -500.0],
                                                 [0.0, 0.0, -0.5, 0.0, 0.0, 3.0]], (9, 99, 199)),
    "one_pixel": ((1, 1), (4, 3), (0, 0), [_rot(30, 1, 1), [0.25, 0.0, 0.0, 0.0, 0.25, 0.0], [1.0, 0.0, 0.0, 0.0, 1.0, 0.0]],
                  (1, 2, 3)),
    "one_row": ((1, 37), (5, 40), (0, 0), [_rot(3, 37, 1), _rot(-90, 37, 1, s=2.0), [1.0, 0.0, -1.5, 0.0, 0.2, 0.0]],
                (0, 0, 0)),
    "larger": ((40, 50), (100, 120), (0, 0), [_rot(15, 50, 40, s=2.2), [0.4, 0.0, 0.0, 0.0, 0.4, 0.0],
                                              [0.5, 0.1, -3.0, -0.1, 0.5, 2.0]], (0, 0, 0)),
    "smaller": ((200, 150), (31, 47), (5, 2), [_rot(-33, 150, 200, s=0.25), [3.0, 0.0, 1.0, 0.0, 6.0, 0.0],
                                               _rot(5, 150, 200)], (0, 0, 0)),
    "crop1280": ((1280, 1280), (512, 512), (384, 384), [rotate_matrix(a, (1280, 1280)) for a in (-10.0, 77.7, 181.5)],
                 (0, 0, 0)),
}


def _images(H, W, content, seed=0):
    """uint8 [B, H, W, 3], a different image per sample."""
    if content == "noise":
        return np.random.default_rng(seed + H * 7919 + W).integers(0, 256, (B, H, W, 3), dtype=np.uint8)
    y = np.arange(H, dtype=np.float32)[:, None, None]
    x = np.arange(W, dtype=np.float32)[None, :, None]
    c = np.arange(3, dtype=np.float32)[None, None, :]
    out = np.empty((B, H, W, 3), np.uint8)
    for i in range(B):
        if content == "gradient":
            v = 0.5 + 0.5 * np.sin(2 * np.pi * ((i + 1) * x / W + (2 - i) * 0.7 * y / H) + c + i)
            out[i] = np.rint(255 * v).astype(np.uint8)
        else:  # all 255, a 0/255 checkerboard, and 2x1 blocks with the channels inverted against each other
            chk = (x // (1 + (i == 2)) + y + (c == 1) * (i == 2)) % 2 == 0
            out[i] = 255 if i == 0 else np.where(chk, 255, 0).astype(np.uint8)
    return out


def _pillow_affine(imgs, mats, size, offset, fill):
    """uint8 [B, H, W, 3] -> uint8 [B, 3, h, w]: Image.transform of each image, cropped at offset."""
    (h, w), (left, top) = size, offset
    out = [np.asarray(Image.fromarray(a).transform((left + w, top + h), Image.AFFINE, list(m), Image.BILINEAR,
                                                   fillcolor=tuple(fill)).crop((left, top, left + w, top + h)))
           for a, m in zip(imgs, mats)]
    return np.ascontiguousarray(np.stack(out).transpose(0, 3, 1, 2))


@functools.lru_cache(maxsize=2)
def _case(name, content):
    (H, W), size, offset, mats, fill = CASES[name]
    imgs = _images(H, W, content)
    return imgs, _pillow_affine(imgs, mats, size, offset, fill)


def _device_input(imgs, layout, device):
    t = torch.from_numpy(imgs)
    return (t if layout == "nhwc" else t.permute(0, 3, 1, 2).contiguous()).to(device)


def _assert_equal(got, ref):
    got, ref = got.cpu(), torch.as_tensor(ref)
    if not torch.equal(got, ref):
        d = (got.int() - ref.int()).abs()
        pytest.fail("%d of %d values differ (max %d), first at %s" %
                    (int((d > 0).sum()), d.numel(), int(d.max()), tuple(torch.nonzero(d)[0].tolist())))


def _captured_rotate_data(im, angle, **kw):
    """(pixels, the AFFINE data Image.rotate passed to Image.transform, or None on a copy / transpose fast path)"""
    cap = {}
    orig = Image.Image.transform

    def spy(self, size, method, data=None, resample=0, fill=1, fillcolor=None):
        cap["a"] = list(data)
        return orig(self, size, method, data, resample, fill, fillcolor)

    Image.Image.transform = spy
    try:
        got = np.asarray(im.rotate(angle, Image.BILINEAR, **kw))
    finally:
        Image.Image.transform = orig
    return got, cap.get("a")


# ---- CPU ------------------------------------------------------------------------------------------------------------
def test_rotate_matrix_is_pillows():
    """rotate_matrix(angle, (W, H), center, translate) == the data Image.rotate hands to Image.transform, over many angles,
    sizes, centres and translations; on Pillow's copy / transpose fast paths it returns the exact quarter-turn matrix,
    whose bilinear transform gives Pillow's pixels."""
    rng = np.random.default_rng(3)
    checked = fast = 0
    for t in range(600):
        W, H = (int(v) for v in rng.integers(1, 40, 2))
        if t % 5 == 0:
            W = H
        angle = float(rng.choice([0.0, 90.0, 180.0, 270.0, -90.0, 360.0, 450.0, -180.0])) if t % 2 == 0 else \
            float(rng.uniform(-720, 720))
        kw = {}
        if t % 4 == 1:
            kw["center"] = (float(rng.uniform(-5, W + 5)), float(rng.uniform(-5, H + 5)))
        elif t % 4 == 2:
            kw["translate"] = (int(rng.integers(-9, 9)), float(rng.uniform(-9, 9)))
        elif t % 4 == 3:
            kw["center"] = (int(rng.integers(0, W + 1)), int(rng.integers(0, H + 1)))
            kw["translate"] = (float(rng.uniform(-5, 5)), 2)
        im = Image.fromarray(rng.integers(0, 256, (H, W, 3), dtype=np.uint8))
        got, data = _captured_rotate_data(im, angle, **kw)
        m = rotate_matrix(angle, (W, H), kw.get("center"), kw.get("translate"))
        if data is not None:
            assert m == data, (angle, W, H, kw)
            checked += 1
        else:
            assert np.array_equal(got, np.asarray(im.transform((W, H), Image.AFFINE, m, Image.BILINEAR))), (angle, W, H)
            fast += 1
    assert checked > 400 and fast > 80


def test_affine_binding_rejects_bad_arguments():
    img = torch.zeros(2, 3, 8, 8, dtype=torch.uint8)
    mats = torch.zeros(2, 6, dtype=torch.float64)
    out = torch.zeros(2, 3, 4, 4, dtype=torch.uint8)
    with pytest.raises(cabi.CcvpeError, match="CUDA tensors"):
        cabi.affine_u8(img, mats, out)
    bad = [
        (dict(img=img.float()), "uint8"),
        (dict(img=torch.zeros(2, 4, 8, 8, dtype=torch.uint8)), "3 channels"),
        (dict(img=torch.zeros(2, 8, 8, 1, dtype=torch.uint8)), "3 channels"),
        (dict(img=torch.zeros(2, 3, 8, 8, dtype=torch.uint8)[..., ::2]), "contiguous"),
        (dict(mats=mats.float()), "float64"),
        (dict(mats=torch.zeros(2, 5, dtype=torch.float64)), "float64"),
        (dict(mats=torch.zeros(3, 6, dtype=torch.float64)), "float64"),
        (dict(mats=torch.zeros(6, 2, dtype=torch.float64).t()), "float64"),
        (dict(out=out.float()), "out must be"),
        (dict(out=torch.zeros(2, 4, 4, 4, dtype=torch.uint8)), "out must be"),
        (dict(out=torch.zeros(2, 3, 0, 4, dtype=torch.uint8)), "empty"),
        (dict(img=torch.zeros(2, 3, 8, 0, dtype=torch.uint8)), "empty"),
        (dict(offset=(-1, 0)), "offset"), (dict(offset=(0, -5)), "offset"), (dict(offset=(1.5, 0)), "offset"),
        (dict(offset=(0,)), "offset"), (dict(offset=(0, 2 ** 31)), "offset"),
        (dict(fill=(0, 0)), "fill"), (dict(fill=(0, 0, 256)), "fill"), (dict(fill=(-1, 0, 0)), "fill"),
        (dict(fill=(0.5, 0, 0)), "fill"), (dict(fill=(0, 0, 0, 0)), "fill"),
        (dict(resample=Image.NEAREST), "bilinear"), (dict(resample=Image.BICUBIC), "bilinear"),
        (dict(resample="nearest"), "bilinear"), (dict(resample=True), "bilinear"),
    ]
    for kw, msg in bad:
        args = dict(img=img, mats=mats, out=out, offset=(0, 0), fill=(0, 0, 0), resample="bilinear")
        args.update(kw)
        with pytest.raises(cabi.CcvpeError, match=msg):
            cabi.affine_u8(args["img"], args["mats"], args["out"], args["offset"], args["fill"], args["resample"])
    for size in [(0, 4), (4, 0), (-1, 4)]:
        with pytest.raises(cabi.CcvpeError, match="positive"):
            affine_u8(img, mats, size)
    with pytest.raises(cabi.CcvpeError, match="out is"):
        affine_u8(img, mats, (5, 4), out=out)
    with pytest.raises(cabi.CcvpeError, match="expand"):
        rotate_u8(img, 10.0, expand=True)
    with pytest.raises(cabi.CcvpeError, match="angles"):
        rotate_u8(img, [1.0, 2.0, 3.0])
    with pytest.raises(cabi.CcvpeError, match="bilinear"):
        rotate_u8(img, 10.0, resample=Image.NEAREST)
    with pytest.raises(cabi.CcvpeError, match="fill"):
        rotate_u8(img, 10.0, fill=(0, 300, 0))


def test_affine_c_abi_rejects_bad_arguments_before_launching():
    """The C entry point checks its arguments itself (the pointers below are never dereferenced)."""
    lib = cabi.load()
    p = ctypes.c_void_p(256)
    fill = (ctypes.c_uint8 * 3)(0, 0, 0)
    bad = [(1, 0, 8, 4, 4, 0, 0), (1, 8, 8, 0, 4, 0, 0), (1, 8, 8, 4, -2, 0, 0), (0, 8, 8, 4, 4, 0, 0),
           (1, -8, 8, 4, 4, 0, 0), (1, 8, 8, 4, 4, -1, 0), (1, 8, 8, 4, 4, 0, -1), (1, 8, 8, 4, 4, 2 ** 31 - 3, 0),
           (70000, 8, 8, 4, 4, 0, 0), (1, 8, 8, 8 * 65536, 4, 0, 0)]
    for nhwc in (0, 1):
        for Bn, H, W, h, w, left, top in bad:
            assert lib.ccvpe_affine_u8(p, nhwc, Bn, H, W, p, h, w, left, top, fill, p, None) != 0, (Bn, H, W, h, w)
            assert b"ccvpe_affine_u8" in lib.ccvpe_last_error()
    assert lib.ccvpe_affine_u8(p, 1, 1, 8, 8, None, 4, 4, 0, 0, fill, p, None) != 0
    assert lib.ccvpe_affine_u8(p, 1, 1, 8, 8, p, 4, 4, 0, 0, None, p, None) != 0


# ---- GPU: bit-exact against Pillow ----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name,content,layout", list(itertools.product(CASES, CONTENTS, ["nhwc", "nchw"])))
def test_affine_matches_pillow(cuda_device, name, content, layout):
    (H, W), size, offset, mats, fill = CASES[name]
    imgs, ref = _case(name, content)
    m = torch.tensor(mats, dtype=torch.float64, device=cuda_device)
    got = affine_u8(_device_input(imgs, layout, cuda_device), m, size, offset, fill)
    assert got.shape == (B, 3) + tuple(size) and got.dtype == torch.uint8 and got.is_contiguous()
    _assert_equal(got, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("hw,angles,kw", [
    ((96, 96), [10.0, -10.0, 33.3], {}),
    ((96, 96), [0.0, 90.0, 270.0], {}),                      # Pillow's copy / transpose fast paths
    ((70, 120), [180.0, 90.0, -90.0], dict(fill=(200, 100, 50))),   # 180 fast path, quarter turns through the transform
    ((70, 120), [360.0, 123.4, -271.0], dict(center=(10, 60.5), translate=(4, -7), fill=(1, 2, 3))),
    ((64, 64), [90.0, 180.0, 0.0], dict(center=(32, 32))),   # a centre given: no fast path, Pillow's rounded matrix
    ((80, 100), [5.0, -5.0, 47.0], dict(translate=(0.5, -2.25))),
])
@pytest.mark.parametrize("layout", ["nhwc", "nchw"])
def test_rotate_matches_pillow(cuda_device, hw, angles, kw, layout):
    imgs = _images(*hw, "noise", seed=5)
    ref = np.stack([np.asarray(Image.fromarray(a).rotate(ang, Image.BILINEAR, center=kw.get("center"),
                                                         translate=kw.get("translate"), fillcolor=kw.get("fill")))
                    for a, ang in zip(imgs, angles)]).transpose(0, 3, 1, 2)
    got = rotate_u8(_device_input(imgs, layout, cuda_device), angles, **kw)
    _assert_equal(got, np.ascontiguousarray(ref))


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["nhwc", "nchw"])
def test_rotate_and_crop_matches_pillow(cuda_device, layout):
    """The aerial augmentation: rotate 1280x1280 images about their centre and keep the central 512x512 (one angle for
    the whole batch here), against Image.rotate(..).crop(box)."""
    imgs = _images(1280, 1280, "gradient", seed=9)
    box = (384, 384, 896, 896)
    ref = np.stack([np.asarray(Image.fromarray(a).rotate(-47.5, Image.BILINEAR).crop(box)) for a in imgs])
    got = rotate_u8(_device_input(imgs, layout, cuda_device), -47.5, size=(512, 512), offset=(384, 384))
    _assert_equal(got, np.ascontiguousarray(ref.transpose(0, 3, 1, 2)))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["rot_any", "one_pixel", "crop1280"])
@pytest.mark.parametrize("layout", ["nhwc", "nchw"])
def test_affine_writes_exactly_its_output(cuda_device, name, layout):
    """out is a view inside a larger sentinel-filled buffer: nothing outside it changes, and every element of it is written
    (two different prefills give the same, correct result)."""
    (H, W), size, offset, mats, fill = CASES[name]
    imgs, ref = _case(name, "noise")
    x = _device_input(imgs, layout, cuda_device)
    m = torch.tensor(mats, dtype=torch.float64, device=cuda_device)
    n, pad = B * 3 * size[0] * size[1], 4099
    results = []
    for sentinel in (0x5A, 0xA5):
        buf = torch.full((pad + n + pad,), sentinel, dtype=torch.uint8, device=cuda_device)
        view = buf[pad:pad + n].view(B, 3, *size)
        assert affine_u8(x, m, size, offset, fill, out=view) is view
        buf = buf.cpu()
        assert bool((buf[:pad] == sentinel).all()) and bool((buf[pad + n:] == sentinel).all()), "write outside out"
        results.append(buf[pad:pad + n].view(B, 3, *size))
    assert torch.equal(results[0], results[1]), "elements of out left unwritten"
    _assert_equal(results[0], ref)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["nhwc", "nchw"])
def test_affine_graph_replay_with_matrices_rewritten(cuda_device, layout):
    """The launch needs no host copy or allocation: captured once in a CUDA graph, then replayed after each in-place
    rewrite of the matrices, it equals an eager call with those matrices (and Pillow)."""
    imgs = _images(300, 260, "gradient", seed=2)
    x = _device_input(imgs, layout, cuda_device)
    size, offset, fill = (200, 180), (30, 40), (10, 20, 30)
    mats = torch.zeros(B, 6, dtype=torch.float64, device=cuda_device)
    out = torch.empty((B, 3) + size, dtype=torch.uint8, device=cuda_device)
    affine_u8(x, mats, size, offset, fill, out=out)            # first launch outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        cabi.affine_u8(x, mats, out, offset, fill)
    rng = np.random.default_rng(4)
    for step in range(4):
        new = [_rot(float(rng.uniform(-180, 180)), 260, 300, s=float(rng.uniform(0.7, 1.4)),
                    tx=float(rng.uniform(-20, 20)), ty=float(rng.uniform(-20, 20))) for _ in range(B)]
        mats.copy_(torch.tensor(new, dtype=torch.float64))
        out.fill_(0)
        graph.replay()
        eager = affine_u8(x, mats, size, offset, fill)
        torch.cuda.synchronize()
        assert torch.equal(out, eager), step
        _assert_equal(out, _pillow_affine(imgs, new, size, offset, fill))


# ---- GPU: end to end ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_model_on_device_rotated_aerials(cuda_device):
    """Aerial tiles rotated on the device give the bf16 model exactly the pixels Pillow's rotation gives it, so all nine
    outputs are identical."""
    g = np.random.default_rng(23)
    grd = torch.from_numpy(g.integers(0, 256, (B, 3, 320, 640), dtype=np.uint8)).to(cuda_device)
    sat = g.integers(0, 256, (B, 512, 512, 3), dtype=np.uint8)
    angles = [12.5, -170.0, 90.0]
    pil_sat = np.stack([np.asarray(Image.fromarray(a).rotate(ang, Image.BILINEAR)) for a, ang in zip(sat, angles)])
    pil_sat = torch.from_numpy(np.ascontiguousarray(pil_sat.transpose(0, 3, 1, 2))).to(cuda_device)
    dev_sat = rotate_u8(torch.from_numpy(sat).to(cuda_device), angles)
    model = build_model("vigor", None, True, 12).to(cuda_device).set_precision("bf16")
    with torch.no_grad():
        a = [t.clone() for t in model(grd, dev_sat)]
        b = model(grd, pil_sat)
    for i, n in enumerate(OUT_NAMES):
        assert torch.equal(a[i], b[i]), n
