"""Drop-in replacements of the reference's four models (reference models.py:49, :346, :655, :954).

Same constructor signatures, same `forward(grd, sat)` 9-tuple, same `state_dict()` keys and shapes (a reference
checkpoint loads with strict=True).  The two EfficientNet-B0 encoders stay PyTorch (`efficientnet.py`); everything
after them runs as sm_100a CUDA kernels through the C ABI (`decoder.PostEncoderPipeline`).  The `nn.Conv2d` /
`nn.ConvTranspose2d` / `nn.Linear` sub-modules below are parameter containers only -- their `forward` is never
called, and there is no PyTorch fallback for the decoder.

Extras over the reference (all optional, defaults reproduce the reference's fp32 behaviour):
  * `set_precision("bf16")`  -- encoders in bf16 channels-last, decoder kernels on tcgen05 tensor cores;
  * `decode_pose(heatmap, ori)` -- the scripts' NumPy argmax/orientation decode as a CUDA kernel;
  * `localize(grd, sat)`     -- forward + decode in one call, returns only the small pose tensors;
  * `resize_u8(img, size)`   -- the reference's bilinear `transforms.Resize` of native-size uint8 images, on the device;
  * `affine_u8(img, matrices, size)`, `rotate_u8(img, angles)` -- Pillow's bilinear affine transform / rotation (+ crop) of
    uint8 images, on the device (augmentation).
"""
from __future__ import annotations

import contextlib
import copy
import math
from typing import Optional

import torch
from torch import nn

from . import cabi
from .decoder import Fork, PostEncoderPipeline, decode_pose
from .efficientnet import EfficientNetB0
from .fast_encoder import FastEncoder
from .specs import KITTI, OXFORD, SKIP_BLOCKS, SKIP_CHANNELS, VIGOR, VariantSpec


def rotate_matrix(angle, size, center=None, translate=None):
    """The AFFINE data `Image.rotate(angle, resample, expand=False, center, translate)` hands to `Image.transform` for an
    image of size = (W, H), in Pillow's own float arithmetic (PIL/Image.py), as a list of 6 floats.  Where Pillow takes a
    copy / transpose fast path instead (angle % 360 in {0, 180}, or {90, 270} on a square image, with neither center nor
    translate given) this returns the exact matrix whose bilinear transform equals that copy / transpose."""
    W, H = size
    angle = angle % 360.0
    if not (center or translate):
        if angle == 0:
            return [1.0, 0.0, 0.0, 0.0, 1.0, 0.0]
        if angle == 180:
            return [-1.0, 0.0, float(W), 0.0, -1.0, float(H)]
        if angle in (90, 270) and W == H:
            return [0.0, -1.0, float(W), 1.0, 0.0, 0.0] if angle == 90 else [0.0, 1.0, 0.0, -1.0, 0.0, float(H)]
    post_trans = (0, 0) if translate is None else translate
    if center is None:
        center = (W / 2, H / 2)
    angle = -math.radians(angle)
    m = [round(math.cos(angle), 15), round(math.sin(angle), 15), 0.0,
         round(-math.sin(angle), 15), round(math.cos(angle), 15), 0.0]
    x, y = -center[0] - post_trans[0], -center[1] - post_trans[1]
    m[2], m[5] = m[0] * x + m[1] * y + m[2], m[3] * x + m[4] * y + m[5]
    m[2] += center[0]
    m[5] += center[1]
    return [float(v) for v in m]


class _Permute(nn.Module):
    """Parameter-free placeholder so that the ground heads keep the reference's Sequential indices (0 and 2)."""

    def __init__(self, *dims):
        super().__init__()
        self.dims = dims

    def forward(self, x):
        return x.permute(*self.dims)


def _double_conv(cin: int, cout: int) -> nn.Sequential:
    return nn.Sequential(nn.Conv2d(cin, cout, 3, padding=1), nn.ReLU(inplace=True), nn.Conv2d(cout, cout, 3, padding=1))


def _final_conv(cout: int) -> nn.Sequential:
    return nn.Sequential(nn.Conv2d(16, 16, 3, padding=1), nn.ReLU(inplace=True), nn.Conv2d(16, cout, 3, padding=1))


class _CVMBase(nn.Module):
    """Builds the parameter tree shared by all four classes from a `VariantSpec`."""

    def __init__(self, spec: VariantSpec, device, circular_padding: bool, ori_noise: Optional[float] = None):
        super().__init__()
        self.device = device                      # stored and unused, exactly like the reference (models.py:52)
        self.circular_padding = circular_padding
        self.spec = spec
        self.grd_efficientnet = EfficientNetB0(circular=bool(circular_padding))
        for l, c in enumerate(spec.head_channels, start=1):
            setattr(self, "grd_feature_to_descriptor%d" % l,
                    nn.Sequential(nn.Conv2d(1280, c, 1), _Permute(0, 2, 3, 1), nn.Conv2d(spec.grd_feat_h, 1, 1),
                                  nn.Flatten(start_dim=1)))
        self.sat_efficientnet = EfficientNetB0(circular=False)
        self.sat_feature_to_descriptors = nn.Sequential(nn.Flatten(start_dim=1), nn.Linear(1280 * 2 * 2, spec.sat_dim))
        self.sat_normalization = nn.Identity()    # parameter-free in the reference too (models.py:106)
        # localisation decoder
        cin = spec.sat_dim
        for i, n in enumerate(range(6, 0, -1)):
            dout = spec.loc_deconv_out[i]
            setattr(self, "deconv%d" % n, nn.ConvTranspose2d(cin + 1, dout, 2, 2))
            if n > 1:
                setattr(self, "conv%d" % n, _double_conv(dout + SKIP_CHANNELS[i], spec.loc_conv_out[i]))
                cin = spec.loc_conv_out[i]
            else:
                self.conv1 = _final_conv(1)
        # orientation decoder
        cin = spec.sat_dim + spec.n_rolls
        for i, n in enumerate(range(6, 0, -1)):
            dout = spec.ori_deconv_out[i]
            setattr(self, "deconv%d_ori" % n, nn.ConvTranspose2d(cin, dout, 2, 2))
            if n > 1:
                setattr(self, "conv%d_ori" % n, _double_conv(dout + SKIP_CHANNELS[i], spec.ori_conv_out[i]))
                cin = spec.ori_conv_out[i]
            else:
                self.conv1_ori = _final_conv(2)
        self._pipeline = [PostEncoderPipeline(self, spec, ori_noise)]   # in a list: not a sub-module, not in state_dict
        self._precision = "fp32"
        self._fast_encoders = [None]                                    # (signature, grd_enc_bf16, sat_enc_bf16)
        self._graphs = [None]                                           # None = eager; dict = CUDA-graph cache
        self._trainer = [None]                                          # training.PostEncoderTrainer, built on first use

    # -- configuration ----------------------------------------------------------------------------------------
    @property
    def pipeline(self) -> PostEncoderPipeline:
        return self._pipeline[0]

    def set_precision(self, precision: str):
        """"fp32": exact reference arithmetic (fp32 encoders, fp32-accumulate CUDA-core decoder kernels).
        "bf16": bf16 channels-last encoders + bf16 decoder kernels with fp32 accumulation (tcgen05 where built)."""
        if precision not in ("fp32", "bf16"):
            raise ValueError("precision must be 'fp32' or 'bf16'")
        self._precision = precision
        self._drop_graphs()
        return self

    def set_backend(self, backend: int):
        self.pipeline.backend = backend
        self._drop_graphs()
        return self

    def set_cuda_graph(self, enabled: bool = True):
        """Serve `forward` from CUDA graphs (one per input shape/dtype): the ~200 kernel launches of a forward are
        captured once and replayed with a single launch, which removes the host launch cost that dominates small
        batches.  Semantics to know: the returned tensors are the graph's static output buffers -- they are overwritten
        by the next `forward` call with the same shapes, so consume (or clone) them first; inputs are copied into
        static device buffers.  Call it again (or load_state_dict / set_precision / .to) after changing weights: the
        cache is dropped.  Eval mode only."""
        self._graphs[0] = {} if enabled else None
        return self

    def _drop_graphs(self):
        if self._graphs[0] is not None:
            self._graphs[0] = {}

    def load_state_dict(self, *args, **kwargs):
        out = super().load_state_dict(*args, **kwargs)
        self._drop_graphs()
        return out

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        if "_graphs" in self.__dict__:
            self._drop_graphs()
        return out

    def train(self, mode: bool = True):
        out = super().train(mode)
        if "_graphs" in self.__dict__:
            self._drop_graphs()
        return out

    def __deepcopy__(self, memo):
        cls = self.__class__
        new = cls.__new__(cls)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            if k in ("_pipeline", "_fast_encoders", "_graphs", "_trainer"):
                continue
            setattr(new, k, copy.deepcopy(v, memo))
        new._pipeline = [PostEncoderPipeline(new, self.spec, self.pipeline.ori_noise)]
        new._pipeline[0].backend = self.pipeline.backend
        new._fast_encoders = [None]
        new._graphs = [None if self._graphs[0] is None else {}]
        new._trainer = [None]
        return new

    # -- encoders (PyTorch) -----------------------------------------------------------------------------------
    def _bf16_encoders(self):
        """Inference execution plans of the two encoders (see fast_encoder.py), rebuilt when encoder weights change."""
        sig = tuple((p.data_ptr(), p._version) for enc in (self.grd_efficientnet, self.sat_efficientnet)
                    for p in list(enc.parameters()) + list(enc.buffers()))
        cached = self._fast_encoders[0]
        if cached is None or cached[0] != sig:
            sat_plan = FastEncoder(self.sat_efficientnet, torch.bfloat16)
            sat_plan.keep = set(SKIP_BLOCKS)            # only the decoder's skips are materialised
            cached = (sig, FastEncoder(self.grd_efficientnet, torch.bfloat16), sat_plan)
            self._fast_encoders[0] = cached
        return cached[1], cached[2]

    def _encode(self, grd, sat):
        """uint8 inputs (an extension over the reference: images as the decoder hands them over) are normalised on the
        device: fused into the stem kernel's loads on the bf16 plan, through `ingest` otherwise."""
        if self._precision == "bf16" and not self.training:
            ge, se = self._bf16_encoders()
            # the two encoders are independent: the ground one runs on a forked side stream (small batches do not fill the GPU)
            fork = Fork(grd.device, enabled=self.pipeline.concurrent and self.pipeline.timer is None)
            with fork:
                fg = ge.extract_features(grd)
            fs, multi = se.extract_features_multiscale(sat)
            fork.join(fg)
            return fg, fs, multi, torch.bfloat16
        if grd.dtype == torch.uint8:
            grd = self.ingest(grd)
        if sat.dtype == torch.uint8:
            sat = self.ingest(sat)
        # fp32 means fp32: cuDNN must not silently drop the encoders to TF32 (torch's default for convolutions)
        cudnn = torch.backends.cudnn           # (keep the caller's benchmark / deterministic choices)
        with cudnn.flags(enabled=True, benchmark=cudnn.benchmark, deterministic=cudnn.deterministic, allow_tf32=False):
            fg = self.grd_efficientnet.extract_features(grd)                      # reference models.py:151
            fs, multi = self.sat_efficientnet.extract_features_multiscale(sat)    # reference models.py:166
        return fg, fs, multi, (torch.bfloat16 if self._precision == "bf16" else torch.float32)

    # -- the reference's entry point --------------------------------------------------------------------------
    def forward(self, grd, sat):
        """Returns (logits_flattened, heatmap, x_ori, matching_score_stacked, ..._stacked2, ..., ..._stacked6)
        with the reference's shapes (models.py:343)."""
        if not (grd.is_cuda and sat.is_cuda):
            raise cabi.CcvpeError("ccvpe_b200 models run on CUDA (sm_100a) only; there is no CPU fallback -- "
                                  "move the model and inputs to a B200")
        if sat.device != grd.device:
            raise cabi.CcvpeError("grd (%s) and sat (%s) must be on the same device" % (grd.device, sat.device))
        if torch.is_grad_enabled() and (grd.requires_grad or sat.requires_grad or
                                        any(p.requires_grad for p in self.parameters())):
            return self._forward_train(grd, sat)           # autograd through the CUDA path (training.py)
        with torch.no_grad(), cabi.device_of(grd):     # kernels / stream / func attributes follow the tensors' device
            if self._graphs[0] is not None and not self.training and self.pipeline.timer is None:
                return self._forward_graphed(grd, sat)
            return self._forward_eager(grd, sat)

    def _forward_train(self, grd, sat):
        """The reference's training forward (train_VIGOR.py:134-135): PyTorch-autograd encoders (train-mode BatchNorm and
        stochastic depth exactly as the reference's), then ONE autograd Function for the whole CUDA post-encoder path whose
        backward runs this library's backward kernels (training.PostEncoderFunction).  Gradients flow to all 98 head /
        decoder parameters, into both encoders, and to `grd` / `sat` if they require grad."""
        from .training import PostEncoderFunction, PostEncoderTrainer
        if self._trainer[0] is None:
            self._trainer[0] = PostEncoderTrainer(self.pipeline)
        if grd.dtype == torch.uint8:
            grd = self.ingest(grd)
        if sat.dtype == torch.uint8:
            sat = self.ingest(sat)
        with cabi.device_of(grd):
            cudnn = torch.backends.cudnn
            bf16 = self._precision == "bf16"
            if bf16:
                # channels-last inputs make cuDNN / ATen run the encoders' convolutions and train-mode BatchNorms in NHWC
                # (measured: 51.8 -> 41.9 ms per B=8 training step); parameters keep their layout
                grd = grd.contiguous(memory_format=torch.channels_last)
                sat = sat.contiguous(memory_format=torch.channels_last)
            # fp32: exact fp32 encoders (no TF32); bf16: mixed precision -- fp32 master weights, bf16 autocast for the
            # encoders' convolutions (BatchNorm statistics stay fp32), bf16 activations / GEMM operands in the CUDA path
            with cudnn.flags(enabled=True, benchmark=cudnn.benchmark, deterministic=cudnn.deterministic, allow_tf32=False), \
                    torch.autocast("cuda", dtype=torch.bfloat16, enabled=bf16):
                fg = self.grd_efficientnet.extract_features(grd)                      # reference models.py:151
                fs, multi = self.sat_efficientnet.extract_features_multiscale(sat)    # reference models.py:166
            dtype = torch.bfloat16 if bf16 else torch.float32
            skips = [multi[i] for i in SKIP_BLOCKS]
            params = list(self.pipeline._params().values())
            return PostEncoderFunction.apply(self._trainer[0], dtype, fg, fs, *skips, *skips, *params)

    def _forward_eager(self, grd, sat):
        fg, fs, multi, dtype = self._encode(grd, sat)
        return self.pipeline.run(fg, fs, multi, dtype)

    def _forward_graphed(self, grd, sat):
        key = (tuple(grd.shape), grd.dtype, tuple(sat.shape), sat.dtype, grd.device.index, self._precision)
        entry = self._graphs[0].get(key)
        if entry is None:
            static_grd, static_sat = torch.empty_like(grd), torch.empty_like(sat)
            static_grd.copy_(grd)
            static_sat.copy_(sat)
            # warm up on a side stream: weight caches, persistent staging buffers, cudaFuncSetAttribute, lazy handles
            side = torch.cuda.Stream(device=grd.device)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    self._forward_eager(static_grd, static_sat)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize(grd.device)
            graph = torch.cuda.CUDAGraph()
            n0 = cabi.launch_count()
            with torch.cuda.graph(graph):
                outs = self._forward_eager(static_grd, static_sat)
            n_captured = cabi.launch_count() - n0
            cabi.add_replayed_launches(-n_captured)          # captured, not executed: keep the executed-launch count honest
            entry = (graph, static_grd, static_sat, outs, n_captured)
            self._graphs[0][key] = entry
        graph, static_grd, static_sat, outs, n_launches = entry
        static_grd.copy_(grd)
        static_sat.copy_(sat)
        graph.replay()
        cabi.add_replayed_launches(n_launches)
        return outs

    # -- extras -----------------------------------------------------------------------------------------------
    @staticmethod
    def decode_pose(heatmap, ori):
        return decode_pose(heatmap, ori)

    @torch.no_grad()
    def localize(self, grd, sat):
        out = self.forward(grd, sat)
        return decode_pose(out[1], out[2])

    @staticmethod
    def ingest(img_u8, shift=None, crop_w=None, out=None):
        """The scripts' input pipeline after image decoding, on the GPU (reference train_VIGOR.py:55-70 ToTensor + ImageNet
        Normalize; datasets.py:118 panorama roll; train_VIGOR.py:272-273 limited-FoV crop): uint8 [B,3,H,W] / [B,H,W,3] ->
        fp32 [B,3,H,crop_w], bit-identical to torchvision's transforms on the same pixels.  `shift`: per-image torch.roll
        shifts along the width (int32 [B] device tensor) or None; `crop_w`: int(W * FoV / 360) or None for the full width."""
        nhwc = img_u8.shape[1] != 3
        B = img_u8.shape[0]
        H, W = (img_u8.shape[1], img_u8.shape[2]) if nhwc else (img_u8.shape[2], img_u8.shape[3])
        if out is None:
            out = torch.empty((B, 3, H, crop_w or W), dtype=torch.float32, device=img_u8.device)
        with cabi.device_of(img_u8):
            cabi.ingest_u8(img_u8, out, shift)
        return out

    @staticmethod
    def resize_u8(img_u8, size, out=None):
        """The reference's transforms.Resize(size) (bilinear) on the GPU: uint8 [B,3,H,W] / [B,H,W,3] -> uint8 [B,3,h,w]
        with size = (h, w), bit-identical to `transforms.Resize(size)` on each image as a PIL image (Pillow's 8-bit
        fixed-point resampler), so everything downstream (`ingest`, `forward` on uint8 images) sees the reference's pixels.
        One call resizes images of one input size: batches whose native sizes differ (KITTI's vary by drive) are grouped by
        size by the caller.  `forward` never resizes; feed it the output of this."""
        h, w = (int(v) for v in size)
        if h <= 0 or w <= 0:
            raise cabi.CcvpeError("resize_u8: size must be two positive ints (h, w), got %r" % (size,))
        if out is None:
            out = torch.empty((img_u8.shape[0], 3, h, w), dtype=torch.uint8, device=img_u8.device)
        elif tuple(out.shape[2:]) != (h, w):
            raise cabi.CcvpeError("resize_u8: out is %s but size is %r" % (tuple(out.shape), (h, w)))
        with cabi.device_of(img_u8):
            cabi.resize_u8(img_u8, out)
        return out

    @staticmethod
    def affine_u8(img_u8, matrices, size, offset=(0, 0), fill=(0, 0, 0), out=None, resample="bilinear"):
        """Pillow's bilinear affine transform on the GPU, one matrix per image: uint8 [B,3,H,W] / [B,H,W,3] -> uint8
        [B,3,h,w] with size = (h, w).  `matrices`: float64 [B,6] on the images' device, each the `data` of
        `Image.transform(.., AFFINE, data, ..)` (output pixel centre -> input coordinate); it is read when the kernel runs,
        so a captured CUDA graph replays with whatever the tensor holds then.  `offset` = (left, top): out[b, :, y, x] is
        pixel (x + left, y + top) of the transform, so the result is bit-identical to
        `Image.transform((left + w, top + h), AFFINE, data, BILINEAR, fillcolor=fill).crop((left, top, left + w, top + h))`
        on each image as a PIL image.  Only bilinear resampling is provided (see INTEGRATION.md)."""
        h, w = (int(v) for v in size)
        if h <= 0 or w <= 0:
            raise cabi.CcvpeError("affine_u8: size must be two positive ints (h, w), got %r" % (size,))
        if out is None:
            out = torch.empty((img_u8.shape[0], 3, h, w), dtype=torch.uint8, device=img_u8.device)
        elif tuple(out.shape[2:]) != (h, w):
            raise cabi.CcvpeError("affine_u8: out is %s but size is %r" % (tuple(out.shape), (h, w)))
        # a CPU tensor reaches the binding, which refuses it with a CcvpeError
        with cabi.device_of(img_u8) if img_u8.is_cuda else contextlib.nullcontext():
            cabi.affine_u8(img_u8, matrices, out, offset, fill, resample)
        return out

    @staticmethod
    def rotate_u8(img_u8, angles, center=None, translate=None, fill=(0, 0, 0), size=None, offset=(0, 0),
                  resample="bilinear", expand=False):
        """Pillow's `Image.rotate(angle, BILINEAR, expand=False, center, translate, fillcolor=fill)` of each image on the GPU,
        bit-identical: uint8 [B,3,H,W] / [B,H,W,3] -> uint8 [B,3,h,w].  `angles`: one angle in degrees (counter-clockwise)
        or one per image; `center` / `translate`: as Pillow's, shared by all images.  size = (h, w) and offset = (left,
        top) fuse a crop: the result is `.crop((left, top, left + w, top + h))` of the rotated image (size None: the input
        size).  The [B,6] matrices are built on the host (`rotate_matrix`) and copied to the device; a CUDA-graph caller
        builds them itself and calls `affine_u8`."""
        if expand:
            raise cabi.CcvpeError("rotate_u8: expand=True is not supported; the output size is the input size or `size`")
        if img_u8.dim() != 4:
            raise cabi.CcvpeError("rotate_u8: img must be a uint8 [B,3,H,W] or [B,H,W,3] tensor")
        B = img_u8.shape[0]
        H, W = (img_u8.shape[2], img_u8.shape[3]) if img_u8.shape[1] == 3 else (img_u8.shape[1], img_u8.shape[2])
        angles = torch.as_tensor(angles, dtype=torch.float64).flatten().tolist()
        if len(angles) == 1:
            angles = angles * B
        if len(angles) != B:
            raise cabi.CcvpeError("rotate_u8: %d angles for %d images" % (len(angles), B))
        mats = torch.tensor([rotate_matrix(a, (W, H), center, translate) for a in angles], dtype=torch.float64)
        return _CVMBase.affine_u8(img_u8, mats.to(img_u8.device), (H, W) if size is None else size, offset, fill,
                                  resample=resample)

    def localize_u8(self, grd_u8, sat_u8, shift=None, crop_w=None, grd_size=None, sat_size=None):
        """uint8 images in, poses out: (resize +) normalise (/ roll / crop) + forward + pose decode, all on the device.
        grd_size / sat_size: (h, w) to resize the native-resolution images to first (`resize_u8`), as the reference's
        Resize does before its roll and crop; None if the images are already at model resolution.  Without a roll or crop
        the bf16 plan reads the uint8 images straight from the stem kernel (no fp32 image is ever materialised)."""
        if grd_size is not None:
            grd_u8 = self.resize_u8(grd_u8, grd_size)
        if sat_size is not None:
            sat_u8 = self.resize_u8(sat_u8, sat_size)
        if shift is None and crop_w is None:
            return self.localize(grd_u8, sat_u8)
        return self.localize(self.ingest(grd_u8, shift, crop_w), sat_u8)


class CVM_VIGOR(_CVMBase):
    """reference models.py:49 -- `CVM_VIGOR(device, circular_padding)`."""

    def __init__(self, device, circular_padding):
        super().__init__(VIGOR, device, circular_padding)


class CVM_VIGOR_ori_prior(_CVMBase):
    """reference models.py:346 -- localisation sweeps only orientations within +-ori_noise (multiples of 18 deg)."""

    #: the matching kernels sweep at most this many orientations per level (24 = +-198 deg; a prior wider than +-180 deg
    #: sweeps orientations twice and carries no information)
    MAX_ROLLS = 24

    def __init__(self, device, ori_noise, circular_padding=True):
        n_rolls = 2 * int(float(ori_noise) / 18) + 1
        if float(ori_noise) < 0 or n_rolls > self.MAX_ROLLS:
            raise ValueError("CVM_VIGOR_ori_prior: ori_noise=%r sweeps %d orientations per level; this implementation "
                             "supports 0 <= ori_noise < %d (at most %d orientations; +-180 deg already covers the full "
                             "circle)" % (ori_noise, n_rolls, 18 * ((self.MAX_ROLLS - 1) // 2 + 1), self.MAX_ROLLS))
        super().__init__(VIGOR, device, circular_padding, ori_noise=float(ori_noise))
        self.ori_noise = ori_noise


class CVM_KITTI(_CVMBase):
    """reference models.py:655 -- `CVM_KITTI(device)`."""

    def __init__(self, device):
        super().__init__(KITTI, device, False)


class CVM_OxfordRobotCar(_CVMBase):
    """reference models.py:954 -- `CVM_OxfordRobotCar(device)`."""

    def __init__(self, device):
        super().__init__(OXFORD, device, False)
