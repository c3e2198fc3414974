"""ctypes binding of libccvpe_b200.so (the C ABI declared in include/ccvpe_b200.h).

There is NO fallback: if the shared library is missing or a call fails, a `CcvpeError` is raised.  torch is used only
to own device memory and the stream; every pointer handed to the library is `tensor.data_ptr()`.
"""
from __future__ import annotations

import ctypes as C
import math
import numbers
import os
from typing import Optional, Sequence

import torch

from . import build as _build

F32, BF16 = 0, 1
ABI_VERSION = 3
SE_SUM_SCALE = 1048576.0    # CCVPE_SE_SUM_SCALE: the squeeze-excite channel sums are int64 fixed point (order independent)
BACKEND_AUTO, BACKEND_SIMT, BACKEND_TCGEN05 = 0, 1, 2

EXPORTED_SYMBOLS = (
    "ccvpe_abi_version", "ccvpe_last_error", "ccvpe_launch_count", "ccvpe_reset_launch_count",
    "ccvpe_grd_descriptor", "ccvpe_grd_descriptors", "ccvpe_igemm", "ccvpe_igemm_plan", "ccvpe_match_scratch_elems", "ccvpe_match_plan", "ccvpe_match_level",
    "ccvpe_softmax_scratch_elems", "ccvpe_softmax_heatmap", "ccvpe_ori_normalize",
    "ccvpe_pose_scratch_bytes", "ccvpe_pose_decode", "ccvpe_bias_silu_nhwc", "ccvpe_dwconv_bias_silu_nhwc", "ccvpe_dwconv_plan",
    "ccvpe_pointwise_silu_nhwc", "ccvpe_stem_conv_silu_nhwc", "ccvpe_se_gate_scale", "ccvpe_mbconv_project_nhwc",
    "ccvpe_wrap_columns_nhwc",
    "ccvpe_ingest_u8", "ccvpe_resize_u8", "ccvpe_affine_u8", "ccvpe_stem_conv_silu_u8_nhwc",
    # training step (config 5)
    "ccvpe_wgrad_workspace_elems", "ccvpe_wgrad", "ccvpe_wgrad_plan", "ccvpe_colsum_workspace_elems", "ccvpe_colsum",
    "ccvpe_relu_bwd", "ccvpe_scale_rows", "ccvpe_planar_to_cl", "ccvpe_cl_to_planar", "ccvpe_ori_normalize_bwd",
    "ccvpe_match_bwd_scratch_elems", "ccvpe_match_level_bwd", "ccvpe_loss_workspace_elems", "ccvpe_infonce_loss",
    "ccvpe_cross_entropy_loss", "ccvpe_orientation_loss", "ccvpe_grd_descriptors_bwd",
    "ccvpe_gt_pyramid", "ccvpe_infonce_loss_binned", "ccvpe_orientation_loss_const", "ccvpe_pose_labels",
    "ccvpe_pose_hypotheses_smem_bytes", "ccvpe_pose_hypotheses", "ccvpe_track_scratch_bytes", "ccvpe_track_step",
)


class CcvpeError(RuntimeError):
    pass


class IgemmDesc(C.Structure):
    """Mirror of `ccvpe_igemm_desc` (include/ccvpe_b200.h)."""
    _fields_ = [
        ("a0", C.c_void_p), ("a1", C.c_void_p),
        ("c0", C.c_int32), ("c1", C.c_int32), ("ld0", C.c_int32), ("ld1", C.c_int32),
        ("B", C.c_int32), ("Hin", C.c_int32), ("Win", C.c_int32), ("Hout", C.c_int32), ("Wout", C.c_int32),
        ("stride", C.c_int32), ("kh", C.c_int32), ("kw", C.c_int32), ("pad", C.c_int32),
        ("N", C.c_int32), ("dtype", C.c_int32),
        ("w_kn", C.c_void_p), ("w_nk", C.c_void_p),
        ("bias", C.c_void_p), ("row_scale", C.c_void_p), ("row_r1", C.c_void_p), ("r1_w", C.c_void_p),
        ("relu", C.c_int32), ("out_mode", C.c_int32), ("out_dtype", C.c_int32), ("ldo", C.c_int32),
        ("out", C.c_void_p),
        ("backend", C.c_int32),
    ]


class WgradDesc(C.Structure):
    """Mirror of `ccvpe_wgrad_desc` (include/ccvpe_b200.h)."""
    _fields_ = [
        ("a0", C.c_void_p), ("a1", C.c_void_p),
        ("c0", C.c_int32), ("c1", C.c_int32), ("ld0", C.c_int32), ("ld1", C.c_int32),
        ("B", C.c_int32), ("Hin", C.c_int32), ("Win", C.c_int32), ("Hout", C.c_int32), ("Wout", C.c_int32),
        ("stride", C.c_int32), ("kh", C.c_int32), ("kw", C.c_int32), ("pad", C.c_int32),
        ("g", C.c_void_p), ("N", C.c_int32), ("ldg", C.c_int32),
        ("g_row_scale", C.c_void_p),
        ("dtype", C.c_int32),
        ("out", C.c_void_p),
        ("workspace", C.c_void_p), ("workspace_elems", C.c_int64),
        ("backend", C.c_int32),
    ]


_lib: Optional[C.CDLL] = None


def lib_path() -> str:
    return _build.LIB_PATH


def load() -> C.CDLL:
    """Loads the in-tree shared library (never builds implicitly: the .so ships with the repo snapshot)."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise CcvpeError("%s not found -- run `python -m ccvpe_b200.build` (or __graft_entry__.build()); "
                         "there is no CPU / PyTorch fallback for the post-encoder path" % path)
    lib = C.CDLL(path)
    lib.ccvpe_abi_version.restype = C.c_int
    lib.ccvpe_last_error.restype = C.c_char_p
    lib.ccvpe_launch_count.restype = C.c_int64
    lib.ccvpe_reset_launch_count.restype = None
    lib.ccvpe_grd_descriptor.restype = C.c_int
    lib.ccvpe_grd_descriptor.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                         C.c_void_p, C.c_void_p, C.c_void_p]
    lib.ccvpe_grd_descriptors.restype = C.c_int
    lib.ccvpe_grd_descriptors.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                          C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int,
                                          C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                          C.POINTER(C.c_void_p), C.POINTER(C.c_int32), C.POINTER(C.c_void_p),
                                          C.c_void_p, C.c_void_p]
    lib.ccvpe_igemm.restype = C.c_int
    lib.ccvpe_igemm.argtypes = [C.POINTER(IgemmDesc), C.c_void_p]
    lib.ccvpe_igemm_plan.restype = C.c_int
    lib.ccvpe_igemm_plan.argtypes = [C.POINTER(IgemmDesc)]
    lib.ccvpe_match_scratch_elems.restype = C.c_int64
    lib.ccvpe_match_scratch_elems.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.ccvpe_match_plan.restype = C.c_int
    lib.ccvpe_match_plan.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int32), C.c_int, C.c_int, C.c_int]
    lib.ccvpe_match_level.restype = C.c_int
    lib.ccvpe_match_level.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                      C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int32), C.c_int, C.c_uint32,
                                      C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_int, C.c_void_p]
    lib.ccvpe_softmax_scratch_elems.restype = C.c_int64
    lib.ccvpe_softmax_scratch_elems.argtypes = [C.c_int, C.c_int64]
    lib.ccvpe_softmax_heatmap.restype = C.c_int
    lib.ccvpe_softmax_heatmap.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p]
    lib.ccvpe_ori_normalize.restype = C.c_int
    lib.ccvpe_ori_normalize.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int64, C.c_void_p]
    lib.ccvpe_pose_scratch_bytes.restype = C.c_int64
    lib.ccvpe_pose_scratch_bytes.argtypes = [C.c_int, C.c_int64]
    lib.ccvpe_pose_decode.restype = C.c_int
    lib.ccvpe_pose_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p]
    lib.ccvpe_pose_hypotheses_smem_bytes.restype = C.c_int64
    lib.ccvpe_pose_hypotheses_smem_bytes.argtypes = [C.c_int, C.c_int]
    lib.ccvpe_pose_hypotheses.restype = C.c_int
    lib.ccvpe_pose_hypotheses.argtypes = [C.c_void_p, C.c_void_p] + [C.c_int] * 5 + [C.c_void_p] * 9
    lib.ccvpe_track_scratch_bytes.restype = C.c_int64
    lib.ccvpe_track_scratch_bytes.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.ccvpe_track_step.restype = C.c_int
    lib.ccvpe_track_step.argtypes = [C.c_void_p] * 3 + [C.c_int] * 3 + [C.c_float] * 2 + [C.c_void_p] * 4
    lib.ccvpe_bias_silu_nhwc.restype = C.c_int
    lib.ccvpe_bias_silu_nhwc.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64,
                                         C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.ccvpe_dwconv_bias_silu_nhwc.restype = C.c_int
    lib.ccvpe_dwconv_bias_silu_nhwc.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int,
                                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                                C.c_void_p, C.c_void_p]
    lib.ccvpe_dwconv_plan.restype = C.c_int
    lib.ccvpe_dwconv_plan.argtypes = [C.c_int] * 6
    lib.ccvpe_pointwise_silu_nhwc.restype = C.c_int
    lib.ccvpe_pointwise_silu_nhwc.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                              C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.ccvpe_stem_conv_silu_nhwc.restype = C.c_int
    lib.ccvpe_stem_conv_silu_nhwc.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                              C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    lib.ccvpe_stem_conv_silu_u8_nhwc.restype = C.c_int
    lib.ccvpe_stem_conv_silu_u8_nhwc.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                                 C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_void_p, C.c_void_p, C.c_int,
                                                 C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    lib.ccvpe_se_gate_scale.restype = C.c_int
    lib.ccvpe_se_gate_scale.argtypes = [C.c_void_p, C.c_float] + [C.c_void_p] * 6 + [C.c_int] * 5 + [C.c_void_p] * 2
    lib.ccvpe_mbconv_project_nhwc.restype = C.c_int
    lib.ccvpe_mbconv_project_nhwc.argtypes = [C.c_void_p] * 6 + [C.c_int] * 4 + [C.c_void_p]
    lib.ccvpe_wrap_columns_nhwc.restype = C.c_int
    lib.ccvpe_wrap_columns_nhwc.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    lib.ccvpe_ingest_u8.restype = C.c_int
    lib.ccvpe_ingest_u8.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                    C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_void_p, C.c_void_p]
    lib.ccvpe_resize_u8.restype = C.c_int
    lib.ccvpe_resize_u8.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                    C.c_void_p]
    lib.ccvpe_affine_u8.restype = C.c_int
    lib.ccvpe_affine_u8.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                    C.c_int, C.POINTER(C.c_uint8), C.c_void_p, C.c_void_p]
    lib.ccvpe_wgrad_workspace_elems.restype = C.c_int64
    lib.ccvpe_wgrad_workspace_elems.argtypes = [C.POINTER(WgradDesc)]
    lib.ccvpe_wgrad.restype = C.c_int
    lib.ccvpe_wgrad.argtypes = [C.POINTER(WgradDesc), C.c_void_p]
    lib.ccvpe_wgrad_plan.restype = C.c_int
    lib.ccvpe_wgrad_plan.argtypes = [C.POINTER(WgradDesc)]
    lib.ccvpe_colsum_workspace_elems.restype = C.c_int64
    lib.ccvpe_colsum_workspace_elems.argtypes = [C.c_int64, C.c_int, C.c_int]
    lib.ccvpe_colsum.restype = C.c_int
    lib.ccvpe_colsum.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                 C.c_void_p, C.c_void_p, C.c_void_p]
    lib.ccvpe_relu_bwd.restype = C.c_int
    lib.ccvpe_relu_bwd.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p]
    lib.ccvpe_scale_rows.restype = C.c_int
    lib.ccvpe_scale_rows.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]
    lib.ccvpe_planar_to_cl.restype = C.c_int
    lib.ccvpe_planar_to_cl.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_void_p]
    lib.ccvpe_cl_to_planar.restype = C.c_int
    lib.ccvpe_cl_to_planar.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_void_p]
    lib.ccvpe_ori_normalize_bwd.restype = C.c_int
    lib.ccvpe_ori_normalize_bwd.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                            C.c_int64, C.c_void_p]
    lib.ccvpe_match_bwd_scratch_elems.restype = C.c_int64
    lib.ccvpe_match_bwd_scratch_elems.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int]
    lib.ccvpe_match_level_bwd.restype = C.c_int
    lib.ccvpe_match_level_bwd.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                          C.POINTER(C.c_int32), C.c_int, C.c_uint32, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                          C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.ccvpe_loss_workspace_elems.restype = C.c_int64
    lib.ccvpe_loss_workspace_elems.argtypes = [C.c_int]
    lib.ccvpe_infonce_loss.restype = C.c_int
    lib.ccvpe_infonce_loss.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p]
    lib.ccvpe_cross_entropy_loss.restype = C.c_int
    lib.ccvpe_cross_entropy_loss.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p]
    lib.ccvpe_orientation_loss.restype = C.c_int
    lib.ccvpe_orientation_loss.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p]
    lib.ccvpe_gt_pyramid.restype = C.c_int
    lib.ccvpe_gt_pyramid.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.ccvpe_infonce_loss_binned.restype = C.c_int
    lib.ccvpe_infonce_loss_binned.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_float,
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.ccvpe_orientation_loss_const.restype = C.c_int
    lib.ccvpe_orientation_loss_const.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p,
                                                 C.c_void_p, C.c_void_p, C.c_void_p]
    lib.ccvpe_pose_labels.restype = C.c_int
    lib.ccvpe_pose_labels.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p]
    lib.ccvpe_grd_descriptors_bwd.restype = C.c_int
    lib.ccvpe_grd_descriptors_bwd.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                              C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int,
                                              C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                              C.POINTER(C.c_int32), C.POINTER(C.c_void_p), C.c_void_p,
                                              C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                              C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p]
    if lib.ccvpe_abi_version() != ABI_VERSION:
        raise CcvpeError("libccvpe_b200.so ABI version mismatch")
    _lib = lib
    return lib


def _check(rc: int, what: str):
    if rc != 0:
        raise CcvpeError("%s failed (%d): %s" % (what, rc, load().ccvpe_last_error().decode()))


def dtype_code(dt: torch.dtype) -> int:
    if dt == torch.float32:
        return F32
    if dt == torch.bfloat16:
        return BF16
    raise CcvpeError("unsupported dtype %s (float32 / bfloat16 only)" % dt)


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _require_cuda(*tensors):
    """Every tensor must live on the CURRENT CUDA device: the library launches on the calling thread's current device and
    on torch's current stream of that device (`_stream`).  The model-level entry points (`forward`, `decode_pose`, ...)
    switch to their tensors' device themselves (`device_of`), so `model.to('cuda:1')` works whatever the current device
    is; direct callers of this binding get a clear error instead of an illegal address."""
    cur = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise CcvpeError("ccvpe_b200 kernels need CUDA tensors (got a %s tensor); there is no CPU fallback"
                             % t.device.type)
        if cur is None:
            cur = torch.cuda.current_device()
        if t.device.index != cur:
            raise CcvpeError("tensor on cuda:%d but the current device is cuda:%d -- wrap the call in "
                             "`with torch.cuda.device(tensor.device):`" % (t.device.index, cur))


def device_of(t: torch.Tensor):
    """Context manager making `t`'s device current (kernels, func attributes and the stream are per device)."""
    return torch.cuda.device(t.device)


_replayed_launches = 0      # kernel launches executed through CUDA-graph replays (the C counter only sees direct launches)


def launch_count() -> int:
    return int(load().ccvpe_launch_count()) + _replayed_launches


def reset_launch_count():
    global _replayed_launches
    _replayed_launches = 0
    load().ccvpe_reset_launch_count()


def add_replayed_launches(n: int):
    global _replayed_launches
    _replayed_launches += int(n)


# ------------------------------------------------------------------------------------------------------------------
# thin typed wrappers (allocate nothing; shapes are the caller's business)
# ------------------------------------------------------------------------------------------------------------------
def grd_descriptor(feat: torch.Tensor, w1, b1, w2, b2, out: torch.Tensor, scratch: torch.Tensor):
    """feat: logical [B, K, H, W] (any strides); out fp32 [B, W*c]."""
    _require_cuda(feat, w1, b1, w2, b2, out, scratch)
    B, K, H, W = feat.shape
    sb, sk, sh, sw = feat.stride()
    c = w1.shape[0]
    _check(load().ccvpe_grd_descriptor(_ptr(feat), dtype_code(feat.dtype), B, K, H, W, sb, sk, sh, sw,
                                       _ptr(w1), _ptr(b1), _ptr(w2), _ptr(b2), c, _ptr(out), _ptr(scratch), _stream()),
           "ccvpe_grd_descriptor")


def grd_descriptors(feat: torch.Tensor, heads, outs, scratch: torch.Tensor):
    """All heads at once.  heads: list of (w1 [c,K], b1 [c], w2 [H], b2 [1]) fp32 tensors; outs: list of fp32 [B, W*c]."""
    B, K, H, W = feat.shape
    sb, sk, sh, sw = feat.stride()
    n = len(heads)
    flat = [t for h in heads for t in h] + list(outs)
    _require_cuda(feat, scratch, *flat)
    arr = lambda ts: (C.c_void_p * n)(*[t.data_ptr() for t in ts])
    cs = (C.c_int32 * n)(*[h[0].shape[0] for h in heads])
    _check(load().ccvpe_grd_descriptors(_ptr(feat), dtype_code(feat.dtype), B, K, H, W, sb, sk, sh, sw, n,
                                        arr([h[0] for h in heads]), arr([h[1] for h in heads]),
                                        arr([h[2] for h in heads]), arr([h[3] for h in heads]), cs, arr(outs),
                                        _ptr(scratch), _stream()), "ccvpe_grd_descriptors")


def igemm(desc: IgemmDesc):
    _check(load().ccvpe_igemm(C.byref(desc), _stream()), "ccvpe_igemm")


IGEMM_KERNELS = ("igemm_simt_kernel", "igemm_tcgen05_kernel", "conv_ring_tcgen05_kernel")


def igemm_kernel_name(desc: IgemmDesc) -> str:
    rc = load().ccvpe_igemm_plan(C.byref(desc))
    if rc < 0:
        _check(rc, "ccvpe_igemm_plan")
    return IGEMM_KERNELS[rc]


def match_scratch_elems(B: int, Cch: int, n_rolls: int) -> int:
    return int(load().ccvpe_match_scratch_elems(B, Cch, n_rolls))


MATCH_KERNELS = ("match_level_simt_kernel", "match_tcgen05_kernel")


def match_kernel_name(dtype: torch.dtype, Cch: int, L: int, offset: int, shifts: Sequence[int], ld_scores_cl: int,
                      backend: int = BACKEND_AUTO) -> str:
    """Which kernel `match_level` launches for this level (bench attribution / tests)."""
    n = len(shifts)
    arr = (C.c_int32 * n)(*[int(s) for s in shifts])
    rc = load().ccvpe_match_plan(dtype_code(dtype), Cch, L, int(offset), arr, n, ld_scores_cl, backend)
    if rc < 0:
        _check(rc, "ccvpe_match_plan")
    return MATCH_KERNELS[rc]


def match_level(x: torch.Tensor, g: torch.Tensor, offset: int, shifts: Sequence[int], max_mask: int,
                scores=None, scores_cl=None, max_out=None, inv_norm=None, xhat=None, scratch=None,
                backend: int = BACKEND_AUTO):
    """x channels-last [B, H, W, C]; g fp32 [B, L]."""
    _require_cuda(x, g, scores, scores_cl, max_out, inv_norm, xhat, scratch)
    B, H, W, Cch = x.shape
    n = len(shifts)
    arr = (C.c_int32 * n)(*[int(s) for s in shifts])
    ld_cl = 0 if scores_cl is None else scores_cl.shape[-1]
    _check(load().ccvpe_match_level(_ptr(x), dtype_code(x.dtype), B, H * W, Cch, _ptr(g), g.shape[1], int(offset), arr,
                                    n, C.c_uint32(max_mask & 0xFFFFFFFF), _ptr(scores), _ptr(scores_cl), ld_cl,
                                    _ptr(max_out), _ptr(inv_norm), _ptr(xhat), _ptr(scratch), backend, _stream()),
           "ccvpe_match_level")


def softmax_heatmap(logits: torch.Tensor, heatmap: torch.Tensor, scratch: torch.Tensor):
    _require_cuda(logits, heatmap, scratch)
    B, n = logits.shape
    _check(load().ccvpe_softmax_heatmap(_ptr(logits), _ptr(heatmap), B, n, _ptr(scratch), _stream()),
           "ccvpe_softmax_heatmap")


def softmax_scratch_elems(B: int, n: int) -> int:
    return int(load().ccvpe_softmax_scratch_elems(B, n))


def ori_normalize(x_cl: torch.Tensor, out: torch.Tensor):
    """x_cl channels-last [B, H, W, ld>=2]; out fp32 [B, 2, H, W]."""
    _require_cuda(x_cl, out)
    B, H, W, ld = x_cl.shape
    _check(load().ccvpe_ori_normalize(_ptr(x_cl), dtype_code(x_cl.dtype), ld, _ptr(out), B, H * W, _stream()),
           "ccvpe_ori_normalize")


def pose_scratch_bytes(B: int, n: int) -> int:
    return int(load().ccvpe_pose_scratch_bytes(B, n))


def pose_decode(heatmap: torch.Tensor, ori: torch.Tensor, idx, rc, cs, angle, valid, scratch):
    _require_cuda(heatmap, ori, idx, rc, cs, angle, valid, scratch)
    B = heatmap.shape[0]
    H, W = heatmap.shape[-2:]
    _check(load().ccvpe_pose_decode(_ptr(heatmap), _ptr(ori), B, H, W, _ptr(idx), _ptr(rc), _ptr(cs), _ptr(angle),
                                    _ptr(valid), _ptr(scratch), _stream()), "ccvpe_pose_decode")


#: the hypothesis counts and disc radii (pixels) `pose_hypotheses` accepts
HYPOTHESES_K = (1, 64)
HYPOTHESES_RADIUS = (0, 32767)


def pose_hypotheses(heatmap: torch.Tensor, ori: torch.Tensor, k: int, radius: int, idx, rc, value, mass, cs, angle,
                    valid, count):
    """The k strongest mutually exclusive modes of each heatmap (include/ccvpe_b200.h, ccvpe_pose_hypotheses), in one
    launch.  heatmap fp32 [B, 1, H, W], ori fp32 [B, 2, H, W]; outputs idx int64 [B, k], rc int32 [B, k, 2], value and
    mass fp32 [B, k], cs fp32 [B, k, 2], angle float64 [B, k], valid uint8 [B, k], count int32 [B].  All contiguous, on the
    current device; every argument is checked before the launch."""
    if not (_is_int(k) and HYPOTHESES_K[0] <= k <= HYPOTHESES_K[1]):
        raise CcvpeError("pose_hypotheses: k must be an int in [%d, %d], got %r" % (*HYPOTHESES_K, k))
    if not (_is_int(radius) and HYPOTHESES_RADIUS[0] <= radius <= HYPOTHESES_RADIUS[1]):
        raise CcvpeError("pose_hypotheses: radius must be an int in [%d, %d] (pixels), got %r"
                         % (*HYPOTHESES_RADIUS, radius))
    _require_f32("heatmap", heatmap, (None, 1, None, None))
    B, _, H, W = heatmap.shape
    if min(B, H, W) <= 0 or B > 65535:
        raise CcvpeError("pose_hypotheses: heatmap must be [B, 1, H, W] with 0 < B <= 65535 and H, W > 0, got %s"
                         % (tuple(heatmap.shape),))
    if load().ccvpe_pose_hypotheses_smem_bytes(H, W) < 0:
        raise CcvpeError("pose_hypotheses: a %dx%d map does not fit the shared memory of one 8-CTA cluster (a band of "
                         "ceil(H/8) + 2 rows per CTA)" % (H, W))
    _require_f32("ori", ori, (B, 2, H, W))
    for name, t, dt, shape in (("idx", idx, torch.int64, (B, k)), ("rc", rc, torch.int32, (B, k, 2)),
                               ("value", value, torch.float32, (B, k)), ("mass", mass, torch.float32, (B, k)),
                               ("cs", cs, torch.float32, (B, k, 2)), ("angle", angle, torch.float64, (B, k)),
                               ("valid", valid, torch.uint8, (B, k)), ("count", count, torch.int32, (B,))):
        if not isinstance(t, torch.Tensor) or t.dtype != dt or tuple(t.shape) != shape or not t.is_contiguous():
            raise CcvpeError("pose_hypotheses: %s must be a contiguous %s tensor of shape %s, got %s %s"
                             % (name, dt, shape, getattr(t, "dtype", type(t).__name__), tuple(getattr(t, "shape", ()))))
    tensors = (heatmap, ori, idx, rc, value, mass, cs, angle, valid, count)
    for name, t in zip(("heatmap", "ori", "idx", "rc", "value", "mass", "cs", "angle", "valid", "count"), tensors):
        if t.data_ptr() % t.element_size():
            raise CcvpeError("pose_hypotheses: %s is misaligned for its dtype" % name)
    _require_cuda(*tensors)
    _check(load().ccvpe_pose_hypotheses(_ptr(heatmap), _ptr(ori), B, H, W, k, radius, _ptr(idx), _ptr(rc), _ptr(value),
                                        _ptr(mass), _ptr(cs), _ptr(angle), _ptr(valid), _ptr(count), _stream()),
           "ccvpe_pose_hypotheses")


#: the process-noise widths (pixels) and uniform-mix weights `track_step` accepts, and its largest map side
TRACK_SIGMA = (0.0, 32.0)
TRACK_EPSILON = (0.0, 1.0)
TRACK_MAX_DIM = 4096


def track_scratch_bytes(B: int, H: int, W: int) -> int:
    return int(load().ccvpe_track_scratch_bytes(B, H, W))


def track_step(belief: torch.Tensor, heatmap: torch.Tensor, motion: torch.Tensor, sigma: float, epsilon: float,
               evidence: torch.Tensor, reset: torch.Tensor, scratch: torch.Tensor):
    """One step of the sequential location filter (include/ccvpe_b200.h, ccvpe_track_step), updating `belief` in place.
    belief and heatmap fp32 [B, 1, H, W] (heatmap's storage must not overlap belief's), motion float64 [B, 6] (read when
    the kernels run), evidence float64 [B], reset uint8 [B], scratch uint8 [>= track_scratch_bytes(B, H, W)].  All
    contiguous, on the current device; sigma in TRACK_SIGMA pixels, epsilon in TRACK_EPSILON; every argument is checked
    before the launch."""
    for name, v, (lo, hi) in (("sigma", sigma, TRACK_SIGMA), ("epsilon", epsilon, TRACK_EPSILON)):
        if not (isinstance(v, numbers.Real) and not isinstance(v, bool) and lo <= v <= hi):
            raise CcvpeError("track_step: %s must be a number in [%g, %g], got %r" % (name, lo, hi, v))
    _require_f32("belief", belief, (None, 1, None, None))
    B, _, H, W = belief.shape
    if not (1 <= B <= 65535 and 1 <= H <= TRACK_MAX_DIM and 1 <= W <= TRACK_MAX_DIM):
        raise CcvpeError("track_step: belief must be [B, 1, H, W] with 1 <= B <= 65535 and 1 <= H, W <= %d, got %s"
                         % (TRACK_MAX_DIM, tuple(belief.shape)))
    _require_f32("heatmap", heatmap, (B, 1, H, W))
    for name, t, dt, shape in (("motion", motion, torch.float64, (B, 6)), ("evidence", evidence, torch.float64, (B,)),
                               ("reset", reset, torch.uint8, (B,))):
        if not isinstance(t, torch.Tensor) or t.dtype != dt or tuple(t.shape) != shape or not t.is_contiguous():
            raise CcvpeError("track_step: %s must be a contiguous %s tensor of shape %s, got %s %s"
                             % (name, dt, shape, getattr(t, "dtype", type(t).__name__), tuple(getattr(t, "shape", ()))))
    need = track_scratch_bytes(B, H, W)
    if not isinstance(scratch, torch.Tensor) or scratch.dtype != torch.uint8 or scratch.dim() != 1 \
            or not scratch.is_contiguous() or scratch.numel() < need:
        raise CcvpeError("track_step: scratch must be a contiguous uint8 tensor of at least %d bytes" % need)
    tensors = (belief, heatmap, motion, evidence, reset, scratch)
    for name, t, align in zip(("belief", "heatmap", "motion", "evidence", "reset", "scratch"), tensors, (4, 4, 8, 8, 1, 8)):
        if t.data_ptr() % align:
            raise CcvpeError("track_step: %s is misaligned (needs %d bytes)" % (name, align))
    b0, h0, nbytes = belief.data_ptr(), heatmap.data_ptr(), belief.numel() * 4
    if b0 < h0 + nbytes and h0 < b0 + nbytes:
        raise CcvpeError("track_step: heatmap overlaps belief; the step writes belief while it reads heatmap")
    _require_cuda(*tensors)
    _check(load().ccvpe_track_step(_ptr(belief), _ptr(heatmap), _ptr(motion), B, H, W, float(sigma), float(epsilon),
                                   _ptr(evidence), _ptr(reset), _ptr(scratch), _stream()), "ccvpe_track_step")


def _check_se_sum(chan_sum: Optional[torch.Tensor]):
    if chan_sum is not None and (chan_sum.dtype != torch.int64 or not chan_sum.is_contiguous()):
        raise CcvpeError("chan_sum must be a contiguous int64 tensor (fixed point, units of 1/SE_SUM_SCALE)")


def bias_silu_nhwc(x: torch.Tensor, bias: Optional[torch.Tensor], y: torch.Tensor, chan_sum: Optional[torch.Tensor] = None):
    """x contiguous NHWC bf16 [B,H,W,C]; y NHWC bf16 view with contiguous channels (any batch/row/pixel strides);
    chan_sum: int64 [B, C] fixed-point accumulator (units of 1/SE_SUM_SCALE), zeroed by the caller."""
    _require_cuda(x, bias, y, chan_sum)
    _check_se_sum(chan_sum)
    B, H, W, Cc = x.shape
    if not x.is_contiguous() or y.stride(3) != 1 or tuple(y.shape) != tuple(x.shape):
        raise CcvpeError("bias_silu_nhwc: x must be contiguous NHWC and y an NHWC view of the same shape")
    _check(load().ccvpe_bias_silu_nhwc(_ptr(x), _ptr(bias), _ptr(y), y.stride(0), y.stride(1), y.stride(2), B, H, W, Cc,
                                       _ptr(chan_sum), _stream()), "ccvpe_bias_silu_nhwc")


def dwconv_bias_silu_nhwc(x_pad: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, y: torch.Tensor, k: int, stride: int,
                          chan_sum: Optional[torch.Tensor] = None):
    """x_pad: pre-padded NHWC bf16 view [B,Hp,Wp,C] (channels contiguous); w bf16 [k*k, C]; y contiguous NHWC bf16."""
    _require_cuda(x_pad, w, bias, y, chan_sum)
    _check_se_sum(chan_sum)
    B, Hp, Wp, Cc = x_pad.shape
    if x_pad.stride(3) != 1 or not y.is_contiguous():
        raise CcvpeError("dwconv_bias_silu_nhwc: channels must be contiguous and y contiguous")
    _check(load().ccvpe_dwconv_bias_silu_nhwc(_ptr(x_pad), x_pad.stride(0), x_pad.stride(1), x_pad.stride(2), Hp, Wp,
                                              _ptr(w), _ptr(bias), _ptr(y), B, Cc, k, stride, _ptr(chan_sum), _stream()),
           "ccvpe_dwconv_bias_silu_nhwc")


DWCONV_KERNELS = ("dwconv_bias_silu_kernel", "dwconv_tile_kernel")


def dwconv_kernel_name(B: int, C: int, Hp: int, Wp: int, k: int, stride: int) -> str:
    """Which kernel `dwconv_bias_silu_nhwc` launches for a [B, Hp, Wp, C] padded input (tests / bench attribution)."""
    rc = load().ccvpe_dwconv_plan(B, C, Hp, Wp, k, stride)
    if rc < 0:
        _check(rc, "ccvpe_dwconv_plan")
    return DWCONV_KERNELS[rc]


def w_nk_layout(per_tap_rows: torch.Tensor, splits: Sequence[int]) -> torch.Tensor:
    """[N, taps, sum(splits)] weights -> bf16 [N, taps, sum(pad(split))], the tcgen05 backend's w_nk layout
    (include/ccvpe_b200.h): every source's K range is zero padded to a multiple of its K-block width, 16 if c <= 16,
    32 if c <= 32, else 64 (the kernels' tc_block_width)."""
    N, taps, _ = per_tap_rows.shape
    pads = [-(-c // kw) * kw for c, kw in ((c, 16 if c <= 16 else (32 if c <= 32 else 64)) for c in splits)]
    out = torch.zeros((N, taps, sum(pads)), dtype=torch.bfloat16, device=per_tap_rows.device)
    src = dst = 0
    for c, cp in zip(splits, pads):
        out[:, :, dst:dst + c] = per_tap_rows[:, :, src:src + c]
        src += c
        dst += cp
    return out


def pad_k_blocks(w: torch.Tensor) -> torch.Tensor:
    """[N, K] weights -> bf16 [N, pad(K)]: the one-source, one-tap case of `w_nk_layout`."""
    return w_nk_layout(w.unsqueeze(1), [w.shape[1]]).squeeze(1)


def pointwise_silu_nhwc(x: torch.Tensor, w_nk: torch.Tensor, bias: Optional[torch.Tensor], out: torch.Tensor,
                        pad_lo: int = 0, pad_hi: int = 0):
    """out[b, lo+h, lo+w, :] = SiLU(x[b,h,w,:] @ W^T + bias).  x: contiguous NHWC bf16 [B,H,W,K]; w_nk = pad_k_blocks(W);
    bias fp32 [N]; out: contiguous bf16 [B, H+lo+hi, W+lo+hi, N] (only its interior is written)."""
    _require_cuda(x, w_nk, bias, out)
    B, H, W, K = x.shape
    N = w_nk.shape[0]
    if not x.is_contiguous() or not out.is_contiguous() or x.dtype != torch.bfloat16 or out.dtype != torch.bfloat16:
        raise CcvpeError("pointwise_silu_nhwc: x and out must be contiguous bf16")
    if tuple(out.shape) != (B, H + pad_lo + pad_hi, W + pad_lo + pad_hi, N):
        raise CcvpeError(f"pointwise_silu_nhwc: out has shape {tuple(out.shape)}")
    if bias is not None and bias.dtype != torch.float32:
        raise CcvpeError("pointwise_silu_nhwc: bias must be fp32")
    _check(load().ccvpe_pointwise_silu_nhwc(_ptr(x), B, H, W, K, K, _ptr(w_nk), _ptr(bias), N, _ptr(out), pad_lo, pad_hi,
                                            _stream()), "ccvpe_pointwise_silu_nhwc")


def stem_conv_silu_nhwc(x: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, out: torch.Tensor, in_pad_lo: int,
                        in_pad_hi: int, out_pad_lo: int, out_pad_hi: int, circular: bool):
    """x: contiguous fp32 NCHW [B,3,H,W]; w fp32 [27, CO] ordered (ci, ky, kx); bias fp32 [CO];
    out: contiguous bf16 [B, Ho+lo+hi, Wo+lo+hi, CO], Ho = (H+in_lo+in_hi-3)//2+1 (interior + wrap columns are written)."""
    _require_cuda(x, w, bias, out)
    B, Cin, H, W = x.shape
    CO = w.shape[1]
    if Cin != 3 or x.dtype != torch.float32 or not x.is_contiguous() or w.dtype != torch.float32 or bias.dtype != torch.float32:
        raise CcvpeError("stem_conv_silu_nhwc: x must be contiguous fp32 [B,3,H,W], w / bias fp32")
    Ho, Wo = (H + in_pad_lo + in_pad_hi - 3) // 2 + 1, (W + in_pad_lo + in_pad_hi - 3) // 2 + 1
    want = (B, Ho + out_pad_lo + out_pad_hi, Wo + out_pad_lo + out_pad_hi, CO)
    if tuple(out.shape) != want or out.dtype != torch.bfloat16 or not out.is_contiguous():
        raise CcvpeError(f"stem_conv_silu_nhwc: out must be contiguous bf16 {want}, got {tuple(out.shape)}")
    _check(load().ccvpe_stem_conv_silu_nhwc(_ptr(x), B, H, W, _ptr(w.contiguous()), _ptr(bias), CO, _ptr(out), in_pad_lo,
                                            in_pad_hi, out_pad_lo, out_pad_hi, 1 if circular else 0, _stream()),
           "ccvpe_stem_conv_silu_nhwc")


def stem_conv_silu_u8_nhwc(x: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, out: torch.Tensor, in_pad_lo: int,
                           in_pad_hi: int, out_pad_lo: int, out_pad_hi: int, circular: bool, crop_w: Optional[int] = None,
                           shift: Optional[torch.Tensor] = None, mean=None, std=None):
    """The stem over a uint8 NCHW image [B,3,H,Wsrc] with ToTensor + Normalize, panorama roll and FoV crop fused into the
    loads.  out: contiguous bf16 [B, Ho+lo+hi, Wo+lo+hi, CO] for the cropped width."""
    _require_cuda(x, w, bias, out, shift)
    B, Cin, H, Wsrc = x.shape
    if Cin != 3 or x.dtype != torch.uint8 or not x.is_contiguous():
        raise CcvpeError("stem_conv_silu_u8_nhwc: x must be contiguous uint8 [B,3,H,W]")
    W = int(crop_w or Wsrc)
    CO = w.shape[1]
    Ho, Wo = (H + in_pad_lo + in_pad_hi - 3) // 2 + 1, (W + in_pad_lo + in_pad_hi - 3) // 2 + 1
    want = (B, Ho + out_pad_lo + out_pad_hi, Wo + out_pad_lo + out_pad_hi, CO)
    if tuple(out.shape) != want or out.dtype != torch.bfloat16 or not out.is_contiguous():
        raise CcvpeError(f"stem_conv_silu_u8_nhwc: out must be contiguous bf16 {want}, got {tuple(out.shape)}")
    if shift is not None and (shift.dtype != torch.int32 or shift.numel() != B):
        raise CcvpeError("stem_conv_silu_u8_nhwc: shift must be int32 [B]")
    m = (C.c_float * 3)(*[float(v) for v in (mean or IMAGENET_MEAN)])
    s = (C.c_float * 3)(*[float(v) for v in (std or IMAGENET_STD)])
    _check(load().ccvpe_stem_conv_silu_u8_nhwc(_ptr(x), B, H, Wsrc, W, _ptr(shift), m, s, _ptr(w.contiguous()), _ptr(bias), CO,
                                               _ptr(out), in_pad_lo, in_pad_hi, out_pad_lo, out_pad_hi, 1 if circular else 0,
                                               _stream()), "ccvpe_stem_conv_silu_u8_nhwc")


def se_gate_scale(chan_sum: torch.Tensor, inv_hw: float, w_red: torch.Tensor, b_red: torch.Tensor, w_se: torch.Tensor,
                  b_se: torch.Tensor, w_proj: torch.Tensor, wg: torch.Tensor, gate_ws: Optional[torch.Tensor] = None,
                  rep: int = 1):
    """wg[b] = w_proj * diag(sigmoid(w_se^T SiLU(w_red mean_b + b_red) + b_se)), mean_b = chan_sum[b] * inv_hw.
    chan_sum int64 fixed point [B, mid]; w_red [R, mid]; w_se [R, mid] (the excite weights transposed); contiguous bf16;
    wg contiguous bf16 [B, rep*cout, rep*mid] (rep > 1: block diagonal, `rep` pixels packed into one GEMM row);
    gate_ws: optional fp32 [B, mid] workspace (required for rep > 1; enables the two-launch form for the deep blocks)."""
    _require_cuda(chan_sum, w_red, b_red, w_se, b_se, w_proj, wg)
    B, mid = chan_sum.shape
    R, cout = w_red.shape[0], w_proj.shape[0]
    for t in (w_red, b_red, w_se, b_se, w_proj, wg):
        if t.dtype != torch.bfloat16 or not t.is_contiguous():
            raise CcvpeError("se_gate_scale: weights, biases and wg must be contiguous bf16")
    if chan_sum.dtype != torch.int64 or not chan_sum.is_contiguous() or tuple(wg.shape) != (B, rep * cout, rep * mid) \
            or tuple(w_red.shape) != (R, mid) or tuple(w_se.shape) != (R, mid) or tuple(w_proj.shape) != (cout, mid):
        raise CcvpeError("se_gate_scale: shape / dtype mismatch")
    if gate_ws is not None:
        _require_cuda(gate_ws)
        if gate_ws.dtype != torch.float32 or not gate_ws.is_contiguous() or gate_ws.numel() < B * mid:
            raise CcvpeError("se_gate_scale: gate_ws must be contiguous fp32 with at least B * mid elements")
    _check(load().ccvpe_se_gate_scale(_ptr(chan_sum), C.c_float(inv_hw), _ptr(w_red), _ptr(b_red), _ptr(w_se), _ptr(b_se),
                                      _ptr(w_proj), _ptr(wg), B, mid, R, cout, int(rep),
                                      _ptr(gate_ws) if gate_ws is not None else None, _stream()), "ccvpe_se_gate_scale")


def mbconv_project_nhwc(d: torch.Tensor, wg: torch.Tensor, residual: Optional[torch.Tensor], out: torch.Tensor,
                        bias: Optional[torch.Tensor] = None, out_biased: Optional[torch.Tensor] = None):
    """out[b] = d[b] @ wg[b]^T (+ residual[b]); optionally out_biased = out + bias (the decoder's skip copy).
    d: contiguous bf16 [B, HW, mid] (or [B, H, W, mid]); wg: [B, cout, mid]; residual / out / out_biased: [B, HW, cout]
    (or [B, H, W, cout]); bias: [cout]."""
    _require_cuda(d, wg, out)
    B, cout, mid = wg.shape
    tensors = [d, wg, out] + [t for t in (residual, bias, out_biased) if t is not None]
    for t in tensors:
        if t.dtype != torch.bfloat16 or not t.is_contiguous():
            raise CcvpeError("mbconv_project_nhwc: operands must be contiguous bf16")
    if d.shape[0] != B or d.shape[-1] != mid or d.numel() % (B * mid) != 0:
        raise CcvpeError("mbconv_project_nhwc: d must be [B, HW, mid]")
    HW = d.numel() // (B * mid)
    for t in (residual, out, out_biased):
        if t is not None and (t.shape[0] != B or t.shape[-1] != cout or t.numel() != B * HW * cout):
            raise CcvpeError("mbconv_project_nhwc: residual / out / out_biased must be [B, HW, cout]")
    if out_biased is not None and (bias is None or bias.numel() != cout):
        raise CcvpeError("mbconv_project_nhwc: out_biased needs a bias of cout elements")
    _check(load().ccvpe_mbconv_project_nhwc(_ptr(d), _ptr(wg), _ptr(residual) if residual is not None else None,
                                            _ptr(bias) if bias is not None else None, _ptr(out),
                                            _ptr(out_biased) if out_biased is not None else None, B, HW, mid, cout,
                                            _stream()), "ccvpe_mbconv_project_nhwc")


def wrap_columns_nhwc(buf: torch.Tensor, H: int, W: int, pad_lo: int, pad_hi: int):
    """Circular width padding inside a contiguous padded NHWC bf16 image [B, H+lo+hi, W+lo+hi, C] (interior already written)."""
    _require_cuda(buf)
    B, Hp, Wp, Cc = buf.shape
    if buf.dtype != torch.bfloat16 or not buf.is_contiguous() or Hp != H + pad_lo + pad_hi or Wp != W + pad_lo + pad_hi:
        raise CcvpeError("wrap_columns_nhwc: buf must be contiguous bf16 [B, H+lo+hi, W+lo+hi, C]")
    _check(load().ccvpe_wrap_columns_nhwc(_ptr(buf), B, H, W, Cc, pad_lo, pad_hi, _stream()), "ccvpe_wrap_columns_nhwc")


# ------------------------------------------------------------------------------------------------------------------
# training step (config 5): backward operators
# ------------------------------------------------------------------------------------------------------------------
WGRAD_KERNELS = ("wgrad_simt_kernel", "wgrad_tcgen05_kernel")


def wgrad(desc: WgradDesc):
    _check(load().ccvpe_wgrad(C.byref(desc), _stream()), "ccvpe_wgrad")


def wgrad_workspace_elems(desc: WgradDesc) -> int:
    n = int(load().ccvpe_wgrad_workspace_elems(C.byref(desc)))
    if n < 0:
        raise CcvpeError("ccvpe_wgrad_workspace_elems: %s" % load().ccvpe_last_error().decode())
    return n


def wgrad_kernel_name(desc: WgradDesc) -> str:
    rc = load().ccvpe_wgrad_plan(C.byref(desc))
    if rc < 0:
        _check(rc, "ccvpe_wgrad_plan")
    return WGRAD_KERNELS[rc]


def colsum(x: torch.Tensor, C_: int, out: torch.Tensor, w: Optional[torch.Tensor] = None, s: int = 1):
    """x channels-last [B, H, W, ld] (first C_ channels); out fp32 [s*s, C_];  out[(y%s)*s + x%s][c] = sum w[b,y/s,x/s] * x."""
    _require_cuda(x, out, w)
    B, H, W, ld = x.shape
    ws = torch.empty(int(load().ccvpe_colsum_workspace_elems(B * H * W, C_, s)), dtype=torch.float32, device=x.device)
    _check(load().ccvpe_colsum(_ptr(x), dtype_code(x.dtype), B, H, W, C_, ld, _ptr(w), s, _ptr(out), _ptr(ws), _stream()),
           "ccvpe_colsum")


def relu_bwd(dh: torch.Tensor, h: torch.Tensor):
    """In place: dh = (h > 0) * dh; both contiguous, same dtype and shape."""
    _require_cuda(dh, h)
    if dh.dtype != h.dtype or dh.shape != h.shape or not dh.is_contiguous() or not h.is_contiguous():
        raise CcvpeError("relu_bwd: dh and h must be contiguous tensors of the same shape and dtype")
    _check(load().ccvpe_relu_bwd(_ptr(dh), _ptr(h), dtype_code(dh.dtype), dh.numel(), _stream()), "ccvpe_relu_bwd")


def scale_rows(x: torch.Tensor, scale: torch.Tensor, y: torch.Tensor):
    """y[..., :] = x[..., :] * scale[...] for contiguous channels-last x / y [.., C] and fp32 scale over the leading dims."""
    _require_cuda(x, scale, y)
    Cc = x.shape[-1]
    if not x.is_contiguous() or not y.is_contiguous() or y.shape != x.shape or scale.dtype != torch.float32 or \
            scale.numel() * Cc != x.numel():
        raise CcvpeError("scale_rows: x, y contiguous [.., C] of the same shape; scale fp32 with one entry per row")
    _check(load().ccvpe_scale_rows(_ptr(x), dtype_code(x.dtype), _ptr(scale), _ptr(y), x.numel() // Cc, Cc, _stream()),
           "ccvpe_scale_rows")


def planar_to_cl(src: torch.Tensor, dst: torch.Tensor):
    """src fp32 planar [B, N, H, W] (or [B, N, HW]) -> dst channels-last [B, H, W, ld] (channels >= N zero filled)."""
    _require_cuda(src, dst)
    B, N = src.shape[0], src.shape[1]
    HW = src.numel() // (B * N)
    if src.dtype != torch.float32 or not src.is_contiguous() or not dst.is_contiguous():
        raise CcvpeError("planar_to_cl: src must be contiguous fp32, dst contiguous")
    _check(load().ccvpe_planar_to_cl(_ptr(src), _ptr(dst), dtype_code(dst.dtype), B, N, HW, dst.shape[-1], _stream()),
           "ccvpe_planar_to_cl")


def cl_to_planar(src: torch.Tensor, n: int, dst: torch.Tensor):
    """src channels-last [B, H, W, ld] (first n channels) -> dst fp32 planar [B, n, H, W]."""
    _require_cuda(src, dst)
    B = src.shape[0]
    HW = src.numel() // (B * src.shape[-1])
    if dst.dtype != torch.float32 or not src.is_contiguous() or not dst.is_contiguous():
        raise CcvpeError("cl_to_planar: dst must be contiguous fp32, src contiguous")
    _check(load().ccvpe_cl_to_planar(_ptr(src), dtype_code(src.dtype), _ptr(dst), B, n, HW, src.shape[-1], _stream()),
           "ccvpe_cl_to_planar")


def ori_normalize_bwd(v_cl: torch.Tensor, d_ori: torch.Tensor, dv: torch.Tensor):
    """v_cl channels-last [B, H, W, ldv]; d_ori fp32 planar [B, 2, H, W]; dv channels-last [B, H, W, ldo]."""
    _require_cuda(v_cl, d_ori, dv)
    B, H, W, ldv = v_cl.shape
    if d_ori.dtype != torch.float32 or not d_ori.is_contiguous() or not dv.is_contiguous() or not v_cl.is_contiguous():
        raise CcvpeError("ori_normalize_bwd: contiguous tensors, d_ori fp32")
    _check(load().ccvpe_ori_normalize_bwd(_ptr(v_cl), dtype_code(v_cl.dtype), ldv, _ptr(d_ori), _ptr(dv),
                                          dtype_code(dv.dtype), dv.shape[-1], B, H * W, _stream()),
           "ccvpe_ori_normalize_bwd")


def match_level_bwd(x: torch.Tensor, g: torch.Tensor, offset: int, shifts: Sequence[int], max_mask: int,
                    scores: torch.Tensor, d_scores, d_scores_cl, d_max, d_xhat, d_xhat2, dx: torch.Tensor, dg: torch.Tensor):
    """x channels-last [B, H, W, C]; g fp32 [B, L]; scores / d_scores fp32 [B, R, H, W]; d_scores_cl, d_max, d_xhat, d_xhat2:
    2-D strided views [B*H*W, >=cols] in x's dtype (last dim contiguous; only the row stride is used) or None."""
    _require_cuda(x, g, scores, d_scores, d_scores_cl, d_max, d_xhat, d_xhat2, dx, dg)
    B, H, W, Cch = x.shape
    n = len(shifts)
    arr = (C.c_int32 * n)(*[int(s) for s in shifts])

    def ld(t):
        if t is None:
            return 0
        if t.dtype != x.dtype or t.stride(-1) != 1:
            raise CcvpeError("match_level_bwd: gradient views must have x's dtype and a contiguous last dim")
        return t.stride(-2)

    scratch = torch.empty(int(load().ccvpe_match_bwd_scratch_elems(B, H * W, Cch, n)), dtype=torch.float32, device=x.device)
    _check(load().ccvpe_match_level_bwd(_ptr(x), dtype_code(x.dtype), B, H * W, Cch, _ptr(g), g.shape[1], int(offset), arr, n,
                                        C.c_uint32(max_mask & 0xFFFFFFFF), _ptr(scores), _ptr(d_scores),
                                        _ptr(d_scores_cl), ld(d_scores_cl), _ptr(d_max), ld(d_max), _ptr(d_xhat), ld(d_xhat),
                                        _ptr(d_xhat2), ld(d_xhat2), _ptr(dx), _ptr(dg), _ptr(scratch), _stream()),
           "ccvpe_match_level_bwd")


def _loss_ws(B: int, device) -> torch.Tensor:
    return torch.empty(int(load().ccvpe_loss_workspace_elems(B)), dtype=torch.float32, device=device)


def infonce_loss(scores: torch.Tensor, labels: torch.Tensor, temperature: float, loss: torch.Tensor, d_scores: torch.Tensor):
    _require_cuda(scores, labels, loss, d_scores)
    B, n = scores.shape
    _check(load().ccvpe_infonce_loss(_ptr(scores), _ptr(labels), B, n, C.c_float(temperature), _ptr(loss), _ptr(d_scores),
                                     _ptr(_loss_ws(B, scores.device)), _stream()), "ccvpe_infonce_loss")


def cross_entropy_loss(logits: torch.Tensor, labels: torch.Tensor, loss: torch.Tensor, d_logits: torch.Tensor):
    _require_cuda(logits, labels, loss, d_logits)
    B, n = logits.shape
    _check(load().ccvpe_cross_entropy_loss(_ptr(logits), _ptr(labels), B, n, _ptr(loss), _ptr(d_logits),
                                           _ptr(_loss_ws(B, logits.device)), _stream()), "ccvpe_cross_entropy_loss")


def orientation_loss(ori: torch.Tensor, gt_ori: torch.Tensor, gt: torch.Tensor, loss: torch.Tensor, d_ori: torch.Tensor):
    _require_cuda(ori, gt_ori, gt, loss, d_ori)
    B = ori.shape[0]
    HW = ori.numel() // (2 * B)
    ws = torch.empty(2048, dtype=torch.float32, device=ori.device)
    _check(load().ccvpe_orientation_loss(_ptr(ori), _ptr(gt_ori), _ptr(gt), B, HW, _ptr(loss), _ptr(d_ori), _ptr(ws),
                                         _stream()), "ccvpe_orientation_loss")


#: max_pool2d kernel sizes of the label pyramid, in the order of the six score volumes a model returns (scores1..6)
GT_PYRAMID_KS = (64, 32, 16, 8, 4, 2)


def _require_f32(name: str, t: torch.Tensor, shape):
    """fp32, contiguous and `shape` (None entries match any size)."""
    if not isinstance(t, torch.Tensor) or t.dtype != torch.float32:
        raise CcvpeError("%s must be a float32 tensor, got %s" % (name, getattr(t, "dtype", type(t).__name__)))
    if t.dim() != len(shape) or any(want is not None and got != want for got, want in zip(t.shape, shape)):
        raise CcvpeError("%s must have shape %s, got %s" % (name, tuple("*" if v is None else v for v in shape),
                                                           tuple(t.shape)))
    if not t.is_contiguous():
        raise CcvpeError("%s must be contiguous" % name)


def gt_pyramid_elems(B: int, H: int, W: int) -> int:
    return sum(B * (H // k) * (W // k) for k in GT_PYRAMID_KS)


def gt_pyramid(gt: torch.Tensor, out: torch.Tensor):
    """gt: fp32 [B, 1, H, W] contiguous, H and W multiples of 64; out: fp32 [gt_pyramid_elems(B, H, W)].  Writes
    max_pool2d(gt, k, stride=k) for k in GT_PYRAMID_KS, each [B, 1, H/k, W/k], one after the other."""
    _require_f32("gt", gt, (None, 1, None, None))
    B, _, H, W = gt.shape
    if B <= 0 or H <= 0 or W <= 0 or H % 64 or W % 64:
        raise CcvpeError("gt_pyramid: H and W must be positive multiples of 64, got gt %s" % (tuple(gt.shape),))
    _require_f32("out", out, (gt_pyramid_elems(B, H, W),))
    _require_cuda(gt, out)
    _check(load().ccvpe_gt_pyramid(_ptr(gt), B, H, W, _ptr(out), _stream()), "ccvpe_gt_pyramid")


def infonce_loss_binned(scores: torch.Tensor, pooled: torch.Tensor, bin_w: torch.Tensor, temperature: float,
                        loss: torch.Tensor, d_scores: torch.Tensor):
    """infonce_loss on the labels pooled[b, 0] * bin_w[b, r] without materialising them: scores fp32 [B, R, h, w],
    pooled fp32 [B, 1, h, w], bin_w fp32 [B, R], loss fp32 [], d_scores fp32 [B, R, h, w]; all contiguous."""
    _require_f32("scores", scores, (None, None, None, None))
    B, R, h, w = scores.shape
    _require_f32("gt_pooled", pooled, (B, 1, h, w))
    _require_f32("bin_weights", bin_w, (B, R))
    _require_f32("loss", loss, ())
    _require_f32("d_scores", d_scores, (B, R, h, w))
    _require_cuda(scores, pooled, bin_w, loss, d_scores)
    _check(load().ccvpe_infonce_loss_binned(_ptr(scores), _ptr(pooled), _ptr(bin_w), B, R, h * w, C.c_float(temperature),
                                            _ptr(loss), _ptr(d_scores), _ptr(_loss_ws(B, scores.device)), _stream()),
           "ccvpe_infonce_loss_binned")


def orientation_loss_const(ori: torch.Tensor, ori_vec: torch.Tensor, gt: torch.Tensor, loss: torch.Tensor,
                           d_ori: torch.Tensor):
    """orientation_loss with the target field ori_vec[b] at every pixel: ori fp32 [B, 2, H, W], ori_vec fp32 [B, 2],
    gt fp32 [B, 1, H, W], loss fp32 [], d_ori fp32 [B, 2, H, W]; all contiguous."""
    _require_f32("ori", ori, (None, 2, None, None))
    B, _, H, W = ori.shape
    _require_f32("ori_vec", ori_vec, (B, 2))
    _require_f32("gt", gt, (B, 1, H, W))
    _require_f32("loss", loss, ())
    _require_f32("d_ori", d_ori, (B, 2, H, W))
    _require_cuda(ori, ori_vec, gt, loss, d_ori)
    ws = torch.empty(2048, dtype=torch.float32, device=ori.device)
    _check(load().ccvpe_orientation_loss_const(_ptr(ori), _ptr(ori_vec), _ptr(gt), B, H * W, _ptr(loss), _ptr(d_ori),
                                               _ptr(ws), _stream()), "ccvpe_orientation_loss_const")


#: the bin counts `pose_labels` accepts: from 10 every bin index of VIGOR's 18-degree rule is a valid tensor index (up to
#: 10 from the end); up to 32 one warp writes a pair's weights
POSE_LABEL_BINS = (10, 32)


def check_pose_label_args(H, W, sigma, n_bins):
    """Raises CcvpeError unless H and W are positive multiples of 64, sigma is a positive finite number and n_bins is an int
    in POSE_LABEL_BINS."""
    if not (_is_int(H) and _is_int(W) and H > 0 and W > 0 and H % 64 == 0 and W % 64 == 0):
        raise CcvpeError("pose_labels: H and W must be positive multiples of 64, got %r x %r" % (H, W))
    if not (isinstance(sigma, numbers.Real) and not isinstance(sigma, bool) and math.isfinite(sigma) and sigma > 0):
        raise CcvpeError("pose_labels: sigma must be a positive finite number, got %r" % (sigma,))
    if not (_is_int(n_bins) and POSE_LABEL_BINS[0] <= n_bins <= POSE_LABEL_BINS[1]):
        raise CcvpeError("pose_labels: n_bins must be an int in [%d, %d], got %r" % (*POSE_LABEL_BINS, n_bins))


def pose_labels(poses: torch.Tensor, sigma: float, n_bins: int, gt: torch.Tensor, pyramid: torch.Tensor,
                bin_weights: torch.Tensor, ori_vec: torch.Tensor):
    """The compact labels of a batch of poses in one launch.  poses: float64 [B, 3] contiguous, rows (row, col, angle_deg),
    read when the kernel runs; gt: fp32 [B, 1, H, W] (H, W multiples of 64), the sigma Gaussian at (row, col) evaluated in
    float64; pyramid: fp32 [gt_pyramid_elems(B, H, W)], as `gt_pyramid` writes it; bin_weights fp32 [B, n_bins] and
    ori_vec fp32 [B, 2], as `losses.orientation_labels` builds them (NaN for an angle outside [0, 360)).  All contiguous,
    on the current device."""
    if not isinstance(poses, torch.Tensor) or poses.dtype != torch.float64 or poses.dim() != 2 or poses.shape[1] != 3 \
            or poses.shape[0] == 0 or not poses.is_contiguous():
        raise CcvpeError("pose_labels: poses must be a contiguous float64 [B, 3] tensor, got %s %s"
                         % (getattr(poses, "dtype", type(poses).__name__), tuple(getattr(poses, "shape", ()))))
    B = poses.shape[0]
    _require_f32("gt", gt, (B, 1, None, None))
    H, W = gt.shape[2], gt.shape[3]
    check_pose_label_args(H, W, sigma, n_bins)
    _require_f32("pyramid", pyramid, (gt_pyramid_elems(B, H, W),))
    _require_f32("bin_weights", bin_weights, (B, n_bins))
    _require_f32("ori_vec", ori_vec, (B, 2))
    _require_cuda(poses, gt, pyramid, bin_weights, ori_vec)
    _check(load().ccvpe_pose_labels(_ptr(poses), B, H, W, float(sigma), n_bins, _ptr(gt), _ptr(pyramid), _ptr(bin_weights),
                                    _ptr(ori_vec), _stream()), "ccvpe_pose_labels")


def grd_descriptors_bwd(feat: torch.Tensor, heads, dgs, dfeat: torch.Tensor, dw1, db1, dw2, db2):
    """Backward of `grd_descriptors`: heads as there; dgs: list of fp32 [B, W*c]; dfeat fp32 [B, K, H, W] contiguous;
    dw1 / db1 / dw2 / db2: lists of fp32 output tensors shaped like the head parameters."""
    B, K, H, W = feat.shape
    sb, sk, sh, sw = feat.stride()
    n = len(heads)
    _require_cuda(feat, dfeat, *[t for h in heads for t in h], *dgs, *dw1, *db1, *dw2, *db2)
    arr = lambda ts: (C.c_void_p * n)(*[t.data_ptr() for t in ts])
    cs = (C.c_int32 * n)(*[h[0].shape[0] for h in heads])
    scratch = torch.empty(2 * n * B * K * W, dtype=torch.float32, device=feat.device)
    _check(load().ccvpe_grd_descriptors_bwd(_ptr(feat), dtype_code(feat.dtype), B, K, H, W, sb, sk, sh, sw, n,
                                            arr([h[0] for h in heads]), arr([h[1] for h in heads]),
                                            arr([h[2] for h in heads]), cs, arr(dgs), _ptr(dfeat), arr(dw1), arr(db1),
                                            arr(dw2), arr(db2), _ptr(scratch), _stream()), "ccvpe_grd_descriptors_bwd")


# ------------------------------------------------------------------------------------------------------------------
# input pipeline (f4)
# ------------------------------------------------------------------------------------------------------------------
IMAGENET_MEAN = (0.485, 0.456, 0.406)      # reference train_VIGOR.py:58, 66
IMAGENET_STD = (0.229, 0.224, 0.225)


def ingest_u8(img: torch.Tensor, out: torch.Tensor, shift: Optional[torch.Tensor] = None, mean=IMAGENET_MEAN,
              std=IMAGENET_STD):
    """img: uint8 [B,3,H,W] (NCHW) or [B,H,W,3] (NHWC), contiguous; out: fp32 [B,3,H,crop_w] contiguous (crop_w <= W);
    shift: int32 [B] device tensor of per-image torch.roll shifts along the width, or None."""
    _require_cuda(img, out, shift)
    if img.dtype != torch.uint8 or not img.is_contiguous() or img.dim() != 4:
        raise CcvpeError("ingest_u8: img must be a contiguous uint8 [B,3,H,W] or [B,H,W,3] tensor")
    nhwc = img.shape[1] != 3
    if nhwc and img.shape[3] != 3:
        raise CcvpeError("ingest_u8: neither dim 1 nor dim 3 has 3 channels")
    B = img.shape[0]
    H, W = (img.shape[1], img.shape[2]) if nhwc else (img.shape[2], img.shape[3])
    if out.dtype != torch.float32 or not out.is_contiguous() or tuple(out.shape[:3]) != (B, 3, H) or out.shape[3] > W:
        raise CcvpeError("ingest_u8: out must be contiguous fp32 [B,3,H,crop_w<=W]")
    if shift is not None and (shift.dtype != torch.int32 or shift.numel() != B):
        raise CcvpeError("ingest_u8: shift must be int32 [B]")
    m = (C.c_float * 3)(*[float(v) for v in mean])
    s = (C.c_float * 3)(*[float(v) for v in std])
    _check(load().ccvpe_ingest_u8(_ptr(img), 1 if nhwc else 0, B, H, W, out.shape[3], _ptr(shift), m, s, _ptr(out), _stream()),
           "ccvpe_ingest_u8")


def resize_u8(img: torch.Tensor, out: torch.Tensor):
    """img: uint8 [B,3,H,W] (NCHW) or [B,H,W,3] (NHWC), contiguous; out: uint8 [B,3,h,w] contiguous.  Writes Pillow's
    bilinear resize of each image to out (bit-identical to transforms.Resize((h, w)) on the image as a PIL image)."""
    if img.dtype != torch.uint8 or not img.is_contiguous() or img.dim() != 4:
        raise CcvpeError("resize_u8: img must be a contiguous uint8 [B,3,H,W] or [B,H,W,3] tensor")
    nhwc = img.shape[1] != 3
    if nhwc and img.shape[3] != 3:
        raise CcvpeError("resize_u8: neither dim 1 nor dim 3 of img %s has 3 channels" % (tuple(img.shape),))
    B = img.shape[0]
    H, W = (img.shape[1], img.shape[2]) if nhwc else (img.shape[2], img.shape[3])
    if out.dtype != torch.uint8 or not out.is_contiguous() or out.dim() != 4 or tuple(out.shape[:2]) != (B, 3):
        raise CcvpeError("resize_u8: out must be a contiguous uint8 [B,3,h,w] tensor")
    h, w = out.shape[2], out.shape[3]
    if min(B, H, W, h, w) <= 0:
        raise CcvpeError("resize_u8: empty image: %s -> %s" % (tuple(img.shape), tuple(out.shape)))
    _require_cuda(img, out)
    _check(load().ccvpe_resize_u8(_ptr(img), 1 if nhwc else 0, B, H, W, h, w, _ptr(out), _stream()), "ccvpe_resize_u8")


#: the resampling filters `affine_u8` accepts: Pillow's BILINEAR (`PIL.Image.Resampling.BILINEAR == 2`), the only one
#: whose affine arithmetic is reproduced exactly
AFFINE_RESAMPLE = ("bilinear", 2)


def _is_int(v) -> bool:
    return isinstance(v, numbers.Integral) and not isinstance(v, bool)


def affine_u8(img: torch.Tensor, matrices: torch.Tensor, out: torch.Tensor, offset: Sequence[int] = (0, 0),
              fill: Sequence[int] = (0, 0, 0), resample="bilinear"):
    """img: uint8 [B,3,H,W] (NCHW) or [B,H,W,3] (NHWC), contiguous; matrices: float64 [B,6] contiguous, on img's device;
    out: uint8 [B,3,h,w] contiguous.  Writes pixel (x + left, y + top) of Pillow's bilinear affine transform of each image
    (`Image.transform(size, AFFINE, matrices[b], BILINEAR, fillcolor=fill)`, bit-identical) to out[b, :, y, x], with
    offset = (left, top)."""
    if isinstance(resample, bool) or resample not in AFFINE_RESAMPLE:
        raise CcvpeError("affine_u8: resample=%r: only bilinear (PIL.Image.BILINEAR) is supported; Pillow's NEAREST and "
                         "BICUBIC affine resamplers are not reproduced" % (resample,))
    if img.dtype != torch.uint8 or not img.is_contiguous() or img.dim() != 4:
        raise CcvpeError("affine_u8: img must be a contiguous uint8 [B,3,H,W] or [B,H,W,3] tensor")
    nhwc = img.shape[1] != 3
    if nhwc and img.shape[3] != 3:
        raise CcvpeError("affine_u8: neither dim 1 nor dim 3 of img %s has 3 channels" % (tuple(img.shape),))
    B = img.shape[0]
    H, W = (img.shape[1], img.shape[2]) if nhwc else (img.shape[2], img.shape[3])
    if matrices.dtype != torch.float64 or not matrices.is_contiguous() or tuple(matrices.shape) != (B, 6):
        raise CcvpeError("affine_u8: matrices must be a contiguous float64 [%d, 6] tensor, got %s %s"
                         % (B, matrices.dtype, tuple(matrices.shape)))
    if out.dtype != torch.uint8 or not out.is_contiguous() or out.dim() != 4 or tuple(out.shape[:2]) != (B, 3):
        raise CcvpeError("affine_u8: out must be a contiguous uint8 [B,3,h,w] tensor")
    h, w = out.shape[2], out.shape[3]
    if min(B, H, W, h, w) <= 0:
        raise CcvpeError("affine_u8: empty image: %s -> %s" % (tuple(img.shape), tuple(out.shape)))
    offset, fill = tuple(offset), tuple(fill)
    if len(offset) != 2 or not all(_is_int(v) and 0 <= v < 2 ** 31 for v in offset):
        raise CcvpeError("affine_u8: offset must be two non-negative ints (left, top), got %r" % (offset,))
    if len(fill) != 3 or not all(_is_int(v) and 0 <= v <= 255 for v in fill):
        raise CcvpeError("affine_u8: fill must be three ints in 0..255 (R, G, B), got %r" % (fill,))
    offset, fill = [int(v) for v in offset], [int(v) for v in fill]
    _require_cuda(img, matrices, out)
    f = (C.c_uint8 * 3)(*fill)
    _check(load().ccvpe_affine_u8(_ptr(img), 1 if nhwc else 0, B, H, W, _ptr(matrices), h, w, offset[0], offset[1], f,
                                  _ptr(out), _stream()), "ccvpe_affine_u8")
