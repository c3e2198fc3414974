"""Device bilinear resize (ccvpe_resize_u8, `model.resize_u8`) against its oracle, Pillow's Image.resize(.., BILINEAR) --
what the reference's transforms.Resize(size) runs on each PIL image.  Every comparison is exact (torch.equal)."""
import ctypes
import functools
import itertools

import numpy as np
import pytest
import torch
from PIL import Image

from ccvpe_b200 import cabi, models
from helpers import OUT_NAMES, build_model

resize_u8 = models.CVM_VIGOR.resize_u8

#: (H, W) -> (h, w): the VIGOR ground and aerial resizes, KITTI-like and Oxford-like targets, down- and upscales, odd and
#: tiny sizes, a 37-tap horizontal kernel (4000 -> 231), a single-axis resize, the identity size, and a 1000x / 1500x
#: downscale (one-pixel tiles whose source window is streamed through shared memory a few rows at a time)
SHAPES = [((1024, 2048), (320, 640)), ((640, 640), (512, 512)), ((375, 1242), (256, 1024)), ((97, 131), (154, 231)),
          ((1200, 1600), (154, 231)), ((333, 777), (320, 640)), ((320, 640), (1024, 2048)), ((5, 3), (7, 2)),
          ((1, 9), (4, 4)), ((3000, 4000), (154, 231)), ((1024, 640), (320, 640)), ((320, 640), (320, 640)),
          ((2000, 3000), (2, 2))]
CONTENTS = ["noise", "gradient", "saturated"]
B = 3


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


def _pillow(imgs, size):
    """uint8 [B, H, W, 3] -> uint8 [B, 3, h, w] through Pillow, image by image."""
    h, w = size
    return np.stack([np.asarray(Image.fromarray(a).resize((w, h), Image.BILINEAR)) for a in imgs]).transpose(0, 3, 1, 2)


@functools.lru_cache(maxsize=2)
def _case(src, dst, content):
    imgs = _images(*src, content)
    return imgs, np.ascontiguousarray(_pillow(imgs, dst))


def _device_input(imgs, layout, device):
    t = torch.from_numpy(imgs)
    return (t if layout == "nhwc" else t.permute(0, 3, 1, 2).contiguous()).to(device)


# ---- CPU ------------------------------------------------------------------------------------------------------------
def test_pillow_oracle_is_the_reference_transform():
    """transforms.Resize([h, w]) on a PIL image is Image.resize((w, h), BILINEAR), the oracle the GPU tests use."""
    import torchvision.transforms as T

    imgs = _images(97, 131, "noise")
    got = np.asarray(T.Resize([154, 231])(Image.fromarray(imgs[0])))
    assert np.array_equal(got.transpose(2, 0, 1), _pillow(imgs[:1], (154, 231))[0])


def test_resize_binding_rejects_bad_arguments():
    img = torch.zeros(1, 3, 8, 8, dtype=torch.uint8)
    out = torch.zeros(1, 3, 4, 4, dtype=torch.uint8)
    with pytest.raises(cabi.CcvpeError, match="CUDA tensors"):
        cabi.resize_u8(img, out)
    with pytest.raises(cabi.CcvpeError, match="uint8"):
        cabi.resize_u8(img.float(), out)
    with pytest.raises(cabi.CcvpeError, match="uint8"):
        cabi.resize_u8(img, out.float())
    with pytest.raises(cabi.CcvpeError, match="3 channels"):
        cabi.resize_u8(torch.zeros(1, 4, 8, 8, dtype=torch.uint8), out)
    with pytest.raises(cabi.CcvpeError, match="out must be"):
        cabi.resize_u8(img, torch.zeros(1, 4, 4, 4, dtype=torch.uint8))
    with pytest.raises(cabi.CcvpeError, match="empty"):
        cabi.resize_u8(img, torch.zeros(1, 3, 0, 4, dtype=torch.uint8))
    with pytest.raises(cabi.CcvpeError, match="empty"):
        cabi.resize_u8(torch.zeros(1, 3, 0, 8, dtype=torch.uint8), out)
    for size in [(0, 4), (4, 0), (-1, 4), (4, -3)]:
        with pytest.raises(cabi.CcvpeError, match="positive"):
            resize_u8(img, size)


def test_resize_c_abi_rejects_bad_sizes_before_launching():
    """The C entry point checks its arguments itself (the pointers below are never dereferenced)."""
    lib = cabi.load()
    p = ctypes.c_void_p(256)
    bad = [(1, 0, 8, 4, 4), (1, 8, 8, 0, 4), (1, 8, 8, 4, -2), (0, 8, 8, 4, 4), (1, -8, 8, 4, 4), (1, 8, 1 << 24, 4, 4),
           # downscales whose coefficient tables alone exceed shared memory, in either axis; 11799470 -> 1 has tables
           # of more than 2^31 bytes for a 32-column tile, which the shared-memory plan must not wrap around
           (1, 8, 8_000_000, 4, 1), (1, 64, 11_799_470, 2, 1), (1, 3000, 4000, 1, 1), (1, 11_799_470, 64, 1, 2)]
    for nhwc in (0, 1):
        for Bn, H, W, h, w in bad:
            assert lib.ccvpe_resize_u8(p, nhwc, Bn, H, W, h, w, p, None) != 0, (Bn, H, W, h, w)
            assert b"ccvpe_resize_u8" in lib.ccvpe_last_error()
    assert b"coefficient tables" in lib.ccvpe_last_error()
    assert lib.ccvpe_resize_u8(None, 1, 1, 8, 8, 4, 4, p, None) != 0


# ---- GPU: bit-exact against Pillow ----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("src,dst,content,layout", [(s, d, c, l) for (s, d), c, l in
                                                    itertools.product(SHAPES, CONTENTS, ["nhwc", "nchw"])])
def test_resize_matches_pillow(cuda_device, src, dst, content, layout):
    imgs, ref = _case(src, dst, content)
    got = resize_u8(_device_input(imgs, layout, cuda_device), dst)
    assert got.shape == (B, 3) + tuple(dst) and got.dtype == torch.uint8 and got.is_contiguous()
    got = got.cpu()
    ref = torch.from_numpy(ref)
    if not torch.equal(got, ref):
        d = (got.int() - ref.int()).abs()
        pytest.fail("%d of %d values differ (max %d), first at %s" %
                    (int((d > 0).sum()), d.numel(), int(d.max()), tuple(torch.nonzero(d)[0].tolist())))


@pytest.mark.gpu
@pytest.mark.parametrize("src,dst", [((97, 131), (154, 231)), ((5, 3), (7, 2)), ((1024, 2048), (320, 640))])
@pytest.mark.parametrize("layout", ["nhwc", "nchw"])
def test_resize_writes_exactly_its_output(cuda_device, src, dst, layout):
    """dst is a view inside a larger sentinel-filled buffer: nothing outside it changes, and every element of it is written
    (two different prefills give the same, correct result)."""
    imgs, ref = _case(src, dst, "noise")
    x = _device_input(imgs, layout, cuda_device)
    n, pad = B * 3 * dst[0] * dst[1], 4099
    results = []
    for fill in (0x5A, 0xA5):
        buf = torch.full((pad + n + pad,), fill, dtype=torch.uint8, device=cuda_device)
        view = buf[pad:pad + n].view(B, 3, *dst)
        assert resize_u8(x, dst, out=view) is view
        buf = buf.cpu()
        assert bool((buf[:pad] == fill).all()) and bool((buf[pad + n:] == fill).all()), "write outside dst"
        results.append(buf[pad:pad + n].view(B, 3, *dst))
    assert torch.equal(results[0], results[1]), "elements of dst left unwritten"
    assert torch.equal(results[0], torch.from_numpy(ref))


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["nhwc", "nchw"])
def test_resize_in_a_cuda_graph(cuda_device, layout):
    """The resize needs no host copy or allocation: captured in a CUDA graph and replayed it equals eager, and two eager
    runs are identical."""
    imgs, ref = _case((1024, 2048), (320, 640), "gradient")
    x = _device_input(imgs, layout, cuda_device)
    eager1 = resize_u8(x, (320, 640)).clone()
    eager2 = resize_u8(x, (320, 640)).clone()
    assert torch.equal(eager1, eager2)
    out = torch.empty_like(eager1)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        cabi.resize_u8(x, out)
    out.fill_(0)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager1)
    assert torch.equal(out.cpu(), torch.from_numpy(ref))


# ---- GPU: end to end ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_models_on_native_size_images(cuda_device, precision):
    """Native-resolution VIGOR images (2048x1024 panoramas, 640x640 aerial tiles) resized on the device give the model
    exactly the pixels Pillow gives it, so every output is identical; likewise localize_u8 with a per-image roll and a
    FoV-180 crop after the resize, as in the reference."""
    g = np.random.default_rng(21)
    grd = g.integers(0, 256, (B, 1024, 2048, 3), dtype=np.uint8)
    sat = g.integers(0, 256, (B, 640, 640, 3), dtype=np.uint8)
    pil_grd = torch.from_numpy(np.ascontiguousarray(_pillow(grd, (320, 640)))).to(cuda_device)
    pil_sat = torch.from_numpy(np.ascontiguousarray(_pillow(sat, (512, 512)))).to(cuda_device)
    grd, sat = torch.from_numpy(grd).to(cuda_device), torch.from_numpy(sat).to(cuda_device)

    model = build_model("vigor", None, True, 12).to(cuda_device).set_precision(precision)
    with torch.no_grad():
        a = model(resize_u8(grd, (320, 640)), resize_u8(sat, (512, 512)))
        a = [t.clone() for t in a]
        b = model(pil_grd, pil_sat)
    for i, n in enumerate(OUT_NAMES):
        assert torch.equal(a[i], b[i]), n

    model = build_model("vigor_prior", 72.0, False, 5).to(cuda_device).set_precision(precision)
    shift = torch.tensor([0, 157, -301], dtype=torch.int32, device=cuda_device)
    crop_w = int(640 * 180 / 360)
    with torch.no_grad():
        pa = model.localize_u8(grd, sat, shift, crop_w, grd_size=(320, 640), sat_size=(512, 512))
        pa = {k: v.clone() for k, v in pa.items()}
        pb = model.localize_u8(pil_grd, pil_sat, shift, crop_w)
    assert pa.keys() == pb.keys()
    for k in pa:                               # angle is NaN where a pose is invalid: NaN == NaN here
        torch.testing.assert_close(pa[k], pb[k], rtol=0, atol=0, equal_nan=True, msg=k)
