"""Every kernel launch of the bf16 encoder plan (fast_encoder.py) against a float64 reference of that launch.

The real models run eagerly (`pipeline.concurrent = False`, no CUDA graph); the `cabi` entry points `FastEncoder.extract`
calls are wrapped (fast_encoder.py resolves `cabi.X` at call time):

  * `stem_conv_silu_nhwc`, `stem_conv_silu_u8_nhwc`  the tcgen05 stem into block 0's padded depthwise input;
  * `pointwise_silu_nhwc`                            the tcgen05 expand 1x1 convs (into a padded buffer) and the head;
  * `wrap_columns_nhwc`                              the circular width padding of the ground encoder;
  * `dwconv_bias_silu_nhwc`                          both depthwise kernels, with the squeeze-excite channel sums;
  * `se_gate_scale`                                  the fused gate kernel and the gate + scale pair;
  * `mbconv_project_nhwc`                            the tcgen05 per-image projection (+ residual, + the decoder's copy);
  * `bias_silu_nhwc`                                 not on this plan (the stem is fused): reaching it is a failure.

Each wrapper calls the original, synchronises and checks the launch at once (the padded staging buffers are shared between
blocks of one shape and are overwritten later).  `FastEncoder.extract` is wrapped too: every launch is attributed to its
(encoder, block), and each block must issue exactly stem or expand (+ wrap) -> depthwise -> SE -> projection, then the head.

References are float64 and start from the operands as the kernel consumes them (bf16 activations and weights, fp32 or bf16
biases, the int64 fixed-point SE sums).  With S the same operation on absolute values, a_ref the pre-activation and
rho = 2^-8 for a bf16 store, an activated output passes if

    |got - silu(a_ref)| <= rho |silu(a_ref)| + 1.1 tau S + EPS_ACT |a_ref| + floor

(1.1 >= max |silu'|; EPS_ACT covers the kernels' SiLU form h + h tanh.approx(h), h = a / 2, whose tanh has a relative error
of about 2^-11 per the PTX ISA; floor = the tensor cores' flush-to-zero allowance, helpers.subnormal_floor).  The
depthwise reference re-pads the STORED interior by the EfficientNet module's rule (TF "same" for stride 2, symmetric for
stride 1, circular width for the ground encoder), so a wrong border or wrap column fails at the launch that reads it.

Every launch is then replayed once into sentinel-filled buffers with guard bands: the guards must be intact, every element
the launch owns must be written (interior, wrap columns, all of y and wg), the padded borders must still hold the sentinel,
and the result must be bit-identical to the plan's own (the SE sums are int64 fixed point: exact even with atomics).

The plan never hands the uint8 stem a roll or a crop (`localize_u8` with a shift or crop ingests to fp32 first); those
paths are checked by `test_stem_conv_silu_u8_fused_ingest` in test_gpu_kernels.py with the same reference.

The CPU self-test at the end shows that the bounds pass a correctly rounded result and fail each planted fault.
"""
import inspect
import math
import time

import numpy as np
import pytest
import torch
from torch.nn import functional as F

from ccvpe_b200 import cabi
from ccvpe_b200.fast_encoder import FastEncoder
from helpers import (RHO_BF16, TINY, bound_check, guard_len, guard_report, guarded, image_subset, sentinel_bits,
                     subnormal_floor)

F64 = torch.float64

#: tau per operator, tau_sum for the SE channel sums, tau_gate for the gate: at least 4x the worst value measured on a B200
#: (1000 W power limit) over every configuration of this file, and never above 1e-4.  Measured worst values:
#:   stem       not measured yet
#:   pointwise  not measured yet
#:   dwconv     not measured yet
#:   project    not measured yet
#:   se_sum     not measured yet
#:   se_gate    not measured yet
TAU = {"stem": 1e-4, "pointwise": 1e-4, "dwconv": 1e-4, "project": 1e-4}
TAU_SUM = 1e-4
TAU_GATE = 1e-4
#: the SiLU approximation: at least 4x the worst (|got - y_ref| - rho |y_ref| - floor) / |a_ref| measured (the whole
#: excess charged to the activation), never above 2^-9.  Measured worst: not measured yet.
EPS_ACT = 2.0 ** -10
SILU_SLOPE = 1.1                 # >= max_a |silu'(a)| = 1.0998
FIX_HALF_ULP = 2.0 ** -21        # one round-to-nearest conversion into the 2^-20 fixed point of the SE sums


# ---------------------------------------------------------------------------------------------------------------
# float64 references
# ---------------------------------------------------------------------------------------------------------------
def silu64(a):
    return a * torch.sigmoid(a)


def act_check(got, a_ref, S, floor, tau):
    """Bound check of an activated bf16 output.  Returns (err/bound, tau needed, eps_act needed)."""
    y = silu64(a_ref)
    ratio, need = bound_check(got, y, SILU_SLOPE * S, RHO_BF16, tau, floor + EPS_ACT * a_ref.abs())
    _, eps_need = bound_check(got, y, a_ref.abs(), RHO_BF16, 0.0, floor)
    return ratio, need, eps_need


def u8_scale_shift(mean, std):
    """(sc, sh) per channel in float32 exactly as ccvpe_stem_conv_silu_u8_nhwc computes them: u8 * sc + sh."""
    f = np.float32
    sc = [f(1.0) / (f(255.0) * f(s)) for s in std]
    sh = [-f(m) / f(s) for m, s in zip(mean, std)]
    return torch.tensor(np.array(sc, np.float32)), torch.tensor(np.array(sh, np.float32))


def stem_operand(x, shift=None, crop_w=None, mean=cabi.IMAGENET_MEAN, std=cabi.IMAGENET_STD):
    """The image as the stem's MMA reads it, float64 [B, 3, H, W]: bf16(x) for fp32 images; for uint8 images the
    per-image torch.roll by `shift`, the crop to `crop_w` columns, then bf16(fp32(u8 * sc + sh)) -- the product and the
    sum are exact in float64 (<= 40 significant bits), so one rounding to fp32 is the kernel's fmaf."""
    if x.dtype != torch.uint8:
        return x.float().to(torch.bfloat16).to(F64)
    if shift is not None:
        x = torch.stack([torch.roll(x[b], int(shift[b]), dims=2) for b in range(x.shape[0])])
    if crop_w:
        x = x[..., :crop_w]
    sc, sh = (t.to(x.device, F64).view(1, 3, 1, 1) for t in u8_scale_shift(mean, std))
    return (x.to(F64) * sc + sh).float().to(torch.bfloat16).to(F64)


def _same_pad(x, lo, hi, circular):
    """NCHW float64: the EfficientNet module's padding (efficientnet.SamePadConv2d): zero rows, circular or zero columns."""
    if circular:
        W = x.shape[3]
        x = torch.cat(([x[..., W - lo:]] if lo else []) + [x] + ([x[..., :hi]] if hi else []), dim=3)
        return F.pad(x, (0, 0, lo, hi))
    return F.pad(x, (lo, hi, lo, hi))


def stem_reference(v, w_taps, bias, lo, hi, circular):
    """v: float64 operand [B, 3, H, W] (`stem_operand`); w_taps fp32 [27, CO] (ci, ky, kx); bias fp32 [CO].
    Returns (a_ref, S, floor) [B, Ho, Wo, CO]."""
    CO = w_taps.shape[1]
    w = w_taps.to(torch.bfloat16).to(F64).t().reshape(CO, 3, 3, 3)
    b = bias.to(F64)
    vp = _same_pad(v, lo, hi, circular)
    a = F.conv2d(vp, w, b, stride=2)
    S = F.conv2d(vp.abs(), w.abs(), b.abs(), stride=2)
    t1 = F.conv2d(vp.abs() + 1, w.abs() + 1, stride=2)
    nhwc = lambda t: t.permute(0, 2, 3, 1)
    return nhwc(a), nhwc(S), nhwc(subnormal_floor(t1) + 4 * TINY)


def pointwise_reference(x, w_nk, bias):
    """1x1 conv of the stored bf16 input [B, H, W, K] with the K-block padded weights w_nk [N, >= K] + fp32 bias.
    Returns (a_ref, S, floor) [B, H, W, N]."""
    B, H, W, K = x.shape
    xa = x.to(F64).reshape(-1, K)
    w = w_nk[:, :K].to(F64)
    b = bias.to(F64)
    a = xa @ w.t() + b
    S = xa.abs() @ w.abs().t() + b.abs()
    floor = subnormal_floor((xa.abs() + 1) @ (w.abs() + 1).t()) + 4 * TINY
    return tuple(t.reshape(B, H, W, -1) for t in (a, S, floor))


def dwconv_reference(interior, w_taps, bias, k, stride, lo, hi, circular):
    """Depthwise conv of the stored interior [B, H, W, C], re-padded by the module's rule; w_taps [k*k, C], bias [C].
    Returns (a_ref, S, floor) [B, Ho, Wo, C]."""
    C = interior.shape[-1]
    x = _same_pad(interior.to(F64).permute(0, 3, 1, 2), lo, hi, circular)
    w = w_taps.to(F64).t().reshape(C, 1, k, k)
    b = bias.to(F64)
    a = F.conv2d(x, w, b, stride=stride, groups=C)
    S = F.conv2d(x.abs(), w.abs(), b.abs(), stride=stride, groups=C)
    t1 = F.conv2d(x.abs() + 1, w.abs() + 1, stride=stride, groups=C)
    nhwc = lambda t: t.permute(0, 2, 3, 1)
    return nhwc(a), nhwc(S), nhwc(subnormal_floor(t1) + 4 * TINY)


def se_sum_conversions(Ho, Wo):
    """Bound on the fixed-point conversions per (b, c) of a depthwise launch: each covers at least one 4-wide output strip
    (a streaming-kernel block owns >= 8 strips of 4 outputs, a tiled-kernel item >= one 8 x 2 micro tile)."""
    return Ho * -(-Wo // 4)


def se_sum_reference(y, n_conv):
    """Per-(b, c) sums of y AS STORED [B, Ho, Wo, C].  Returns (ref, S, floor) [B, C]."""
    y64 = y.to(F64)
    return y64.sum(dim=(1, 2)), y64.abs().sum(dim=(1, 2)), n_conv * FIX_HALF_ULP


def se_gate_reference(sums, hw, w_red, b_red, w_se_t, b_se, w_proj):
    """From the int64 sums as stored: mean = sums 2^-20 / hw, h = silu(W_red mean + b_red), g = sigmoid(W_se h + b_se),
    wg = w_proj diag(g).  Returns (g [B, mid], wg [B, cout, mid])."""
    mean = sums.to(F64) / cabi.SE_SUM_SCALE / hw
    h = silu64(mean @ w_red.to(F64).t() + b_red.to(F64))
    g = torch.sigmoid(h @ w_se_t.to(F64) + b_se.to(F64))
    return g, w_proj.to(F64).unsqueeze(0) * g.unsqueeze(1)


def project_reference(d, wg, residual=None):
    """d [B, HW, mid] @ wg[b]^T (+ residual [B, HW, cout]).  Returns (ref, S, floor) [B, HW, cout]."""
    d64, w = d.to(F64), wg.to(F64)
    ref = torch.bmm(d64, w.transpose(1, 2))
    S = torch.bmm(d64.abs(), w.abs().transpose(1, 2))
    floor = subnormal_floor(torch.bmm(d64.abs() + 1, w.abs().transpose(1, 2) + 1)) + 4 * TINY
    if residual is not None:
        r = residual.to(F64)
        ref, S = ref + r, S + r.abs()
    return ref, S, floor


def unpack_rep(t, rep, n):
    """[B, P / rep, rep * n] packed rows (rep pixels per GEMM row) -> [B, P, n]."""
    return t.reshape(t.shape[0], -1, n)


# ---------------------------------------------------------------------------------------------------------------
# the recorder
# ---------------------------------------------------------------------------------------------------------------
ENTRIES = ("stem_conv_silu_nhwc", "stem_conv_silu_u8_nhwc", "pointwise_silu_nhwc", "wrap_columns_nhwc",
           "dwconv_bias_silu_nhwc", "se_gate_scale", "mbconv_project_nhwc", "bias_silu_nhwc")
_ORIG = {e: getattr(cabi, e) for e in ENTRIES}
_ORIG_EXTRACT = FastEncoder.extract
FEATURES = set()              # what the checked launches reached (see test_every_encoder_kernel_was_checked)
CONFIGS_RUN = set()
MEASURED = {}                 # operator -> worst tau (or eps_act) needed over the file


def _written_mask(shape, lo, H, W, wrap):
    """bool [B, Hp, Wp, C]: the interior rows lo..lo+H, columns lo..lo+W, plus every column of those rows if `wrap`."""
    m = torch.zeros(shape, dtype=torch.bool)
    if wrap:
        m[:, lo:lo + H] = True
    else:
        m[:, lo:lo + H, lo:lo + W] = True
    return m


class Recorder:
    def __init__(self, monkeypatch, model):
        self.model = model
        self.rows = []            # (entry, where, kernel, geometry, worst err/bound, tau needed)
        self.failures = []
        self.intercepted = dict.fromkeys(ENTRIES, 0)
        self.checked = dict.fromkeys(ENTRIES, 0)
        self.ctx = None
        self.extracts = 0
        self._install(monkeypatch)

    # -- bookkeeping ---------------------------------------------------------------------------------------------
    def _record(self, entry, kernel, geom, results, problems=()):
        """results: list of (name, ratio, need, operator)"""
        where = "%s/%s" % (self.ctx["enc"], self.ctx["block"])
        for name, ratio, nd, op in results:
            MEASURED[op] = max(MEASURED.get(op, 0.0), nd)
            if not ratio <= 1.0:
                self.failures.append("%s %s [%s, %s] %s: err/bound %.3g (%s would need %.3g)" % (
                    entry, where, kernel, geom, name, ratio, op, nd))
        for p in problems:
            self.failures.append("%s %s [%s, %s] %s" % (entry, where, kernel, geom, p))
        self.rows.append((entry, where, kernel, geom, max([r[1] for r in results] + [0.0]),
                          max([r[2] for r in results if not r[3].startswith("eps")] + [0.0])))
        self.checked[entry] += 1

    def _fail(self, entry, what):
        where = "?" if self.ctx is None else "%s/%s" % (self.ctx["enc"], self.ctx["block"])
        self.failures.append("%s %s: %s" % (entry, where, what))

    # -- wrappers --------------------------------------------------------------------------------------------------
    def _install(self, mp):
        rec = self
        ge_mod, se_mod = self.model.grd_efficientnet, self.model.sat_efficientnet

        def extract(fe, x, keep_blocks):
            ge, se = rec.model._bf16_encoders()
            name, enc = ("grd", ge_mod) if fe is ge else ("sat", se_mod)
            assert fe is ge or fe is se
            rec.ctx = dict(enc=name, module=enc, fe=fe, block="stem", seq=[], circular=bool(enc._conv_stem._circular))
            try:
                res = _ORIG_EXTRACT(fe, x, keep_blocks)
            finally:
                ctx, rec.ctx = rec.ctx, None
            rec.extracts += 1
            expect = [("stem", "stem")]
            for i, blk in enumerate(enc._blocks):
                if blk._has_expand:
                    expect.append(("pw", i))
                    if ctx["circular"]:
                        expect.append(("wrap", i))
                expect += [("dw", i), ("se", i), ("proj", i)]
            expect.append(("pw", "head"))
            if ctx["seq"] != expect:
                rec.failures.append("%s encoder issued %s, expected %s" % (name, ctx["seq"], expect))
            return res

        mp.setattr(FastEncoder, "extract", extract)
        checks = {"stem_conv_silu_nhwc": ("stem", self.check_stem), "stem_conv_silu_u8_nhwc": ("stem", self.check_stem),
                  "pointwise_silu_nhwc": ("pw", self.check_pointwise), "wrap_columns_nhwc": ("wrap", self.check_wrap),
                  "dwconv_bias_silu_nhwc": ("dw", self.check_dwconv), "se_gate_scale": ("se", self.check_se),
                  "mbconv_project_nhwc": ("proj", self.check_project), "bias_silu_nhwc": ("bias_silu", None)}

        def make(entry):
            orig = _ORIG[entry]
            sig = inspect.signature(orig)
            step, check = checks[entry]

            def wrapper(*args, **kwargs):
                rec.intercepted[entry] += 1
                ba = sig.bind(*args, **kwargs)
                ba.apply_defaults()
                a = dict(ba.arguments)
                if entry == "se_gate_scale" and a["gate_ws"] is not None:
                    a["gate_ws"].fill_(float("nan"))          # shows whether the two-launch form wrote it
                orig(*args, **kwargs)
                torch.cuda.synchronize()
                if rec.ctx is None:
                    rec._fail(entry, "launched outside FastEncoder.extract")
                    return
                if check is None:
                    rec._fail(entry, "is not on the bf16 encoder plan (the stem is fused)")
                    return
                ctx = rec.ctx
                if step == "pw":
                    nxt = 0 if ctx["block"] == "stem" else ctx["block"] + 1
                    ctx["block"] = nxt if nxt < len(ctx["module"]._blocks) else "head"
                elif step == "dw" and ctx["seq"] and ctx["seq"][-1][0] == "stem":
                    ctx["block"] = 0
                ctx["seq"].append((step, ctx["block"]))
                check(entry, a)

            mp.setattr(cabi, entry, wrapper)

        for e in ENTRIES:
            make(e)

    # -- checks ----------------------------------------------------------------------------------------------------
    def check_stem(self, entry, a):
        enc, ctx = self.ctx["module"], self.ctx
        x, out = a["x"], a["out"]
        stem, dw0 = enc._conv_stem, enc._blocks[0]._depthwise_conv
        lo, hi, olo, ohi, circ = stem._pad_lo, stem._pad_hi, dw0._pad_lo, dw0._pad_hi, ctx["circular"]
        if (a["in_pad_lo"], a["in_pad_hi"], a["out_pad_lo"], a["out_pad_hi"], bool(a["circular"])) != (lo, hi, olo, ohi, circ):
            self._fail(entry, "padding / wrap arguments differ from the encoder module's")
        u8 = entry.endswith("u8_nhwc")
        shift, crop_w = (a["shift"], a["crop_w"]) if u8 else (None, None)
        B = x.shape[0]
        sub = image_subset(B)
        v = stem_operand(x[sub], None if shift is None else shift[sub], crop_w, a.get("mean") or cabi.IMAGENET_MEAN,
                         a.get("std") or cabi.IMAGENET_STD)
        a_ref, S, floor = stem_reference(v, a["w"], a["bias"], lo, hi, circ)
        Ho, Wo = a_ref.shape[1:3]
        o = out[sub]
        r = act_check(o[:, olo:olo + Ho, olo:olo + Wo], a_ref, S, floor, TAU["stem"])
        res = [("out", r[0], r[1], "stem"), ("out", r[0], r[2], "eps_act")]
        written = _written_mask(o.shape, olo, Ho, Wo, circ).to(o.device)
        problems = []
        if circ:
            rows = o[:, olo:olo + Ho]
            if olo and not torch.equal(rows[:, :, :olo], rows[:, :, Wo:Wo + olo]):
                problems.append("left wrap columns differ from interior columns [Wo - lo, Wo)")
            if ohi and not torch.equal(rows[:, :, olo + Wo:], rows[:, :, olo:olo + ohi]):
                problems.append("right wrap columns differ from interior columns [0, hi)")
        if not bool((o[~written] == 0).all()):
            problems.append("wrote %d elements outside the interior / wrap columns" % int((o[~written] != 0).sum()))
        problems += self._replay(entry, a, "out", written=_written_mask(out.shape, olo, Ho, Wo, circ).to(out.device))
        kind = "u8" if u8 else "fp32"
        FEATURES.add(("stem", kind, circ))
        geom = "B%d %dx%d->%dx%d %s%s%s" % (B, x.shape[2], x.shape[3], Ho, Wo, kind, " circular" if circ else "",
                                            "" if shift is None else " rolled")
        self._record(entry, "stem_tcgen05_kernel", geom, res, problems)

    def check_pointwise(self, entry, a):
        ctx = self.ctx
        x, out, lo, hi = a["x"], a["out"], a["pad_lo"], a["pad_hi"]
        B, H, W, K = x.shape
        if ctx["block"] != "head":
            dw = ctx["module"]._blocks[ctx["block"]]._depthwise_conv
            if (lo, hi) != (dw._pad_lo, dw._pad_hi):
                self._fail(entry, "padding (%d, %d) differs from the depthwise conv's (%d, %d)" % (lo, hi, dw._pad_lo,
                                                                                                  dw._pad_hi))
        sub = image_subset(B)
        a_ref, S, floor = pointwise_reference(x[sub], a["w_nk"], a["bias"])
        o = out[sub]
        got = o[:, lo:lo + H, lo:lo + W]
        r = act_check(got, a_ref, S, floor, TAU["pointwise"])
        res = [("out", r[0], r[1], "pointwise"), ("out", r[0], r[2], "eps_act")]
        problems = []
        # the border must be exactly 0; in the circular encoder the wrap columns are checked after wrap_columns_nhwc
        border = ~_written_mask(o.shape, lo, H, W, ctx["circular"]).to(o.device)
        if not bool((o[border] == 0).all()):
            problems.append("%d border elements are not 0" % int((o[border] != 0).sum()))
        problems += self._replay(entry, a, "out", written=_written_mask(out.shape, lo, H, W, False).to(out.device))
        N = out.shape[-1]
        geom = "B%d %dx%d K=%d N=%d pad=(%d,%d)" % (B, H, W, K, N, lo, hi)
        self._record(entry, "igemm_tcgen05_kernel", geom, res, problems)

    def check_wrap(self, entry, a):
        buf, H, W, lo, hi = a["buf"], a["H"], a["W"], a["pad_lo"], a["pad_hi"]
        dw = self.ctx["module"]._blocks[self.ctx["block"]]._depthwise_conv
        problems = []
        if (lo, hi) != (dw._pad_lo, dw._pad_hi):
            problems.append("padding (%d, %d) differs from the depthwise conv's" % (lo, hi))
        o = buf[image_subset(buf.shape[0])]
        rows = o[:, lo:lo + H]
        if lo and not torch.equal(rows[:, :, :lo], rows[:, :, W:W + lo]):
            problems.append("left wrap columns differ from interior columns [W - lo, W)")
        if hi and not torch.equal(rows[:, :, lo + W:], rows[:, :, lo:lo + hi]):
            problems.append("right wrap columns differ from interior columns [0, hi)")
        if not (bool((o[:, :lo] == 0).all()) and bool((o[:, lo + H:] == 0).all())):
            problems.append("the zero rows above / below the image are not 0")
        FEATURES.add(("wrap",))
        self._record(entry, "wrap_columns_kernel", "B%d %dx%d C=%d pad=(%d,%d)" % (buf.shape[0], H, W, buf.shape[3], lo, hi),
                     [("buf", 0.0, 0.0, "wrap")], problems)

    def check_dwconv(self, entry, a):
        ctx = self.ctx
        blk = ctx["module"]._blocks[ctx["block"]]
        dwm = blk._depthwise_conv
        xp, y, sums, k, s = a["x_pad"], a["y"], a["chan_sum"], a["k"], a["stride"]
        lo, hi = dwm._pad_lo, dwm._pad_hi
        if (k, s) != (dwm.kernel_size[0], dwm.stride[0]):
            self._fail(entry, "k%d s%d differ from the module's" % (k, s))
        B, Hp, Wp, C = xp.shape
        H, W = Hp - lo - hi, Wp - lo - hi
        Ho, Wo = y.shape[1:3]
        ctx["hw"] = Ho * Wo
        kernel = cabi.dwconv_kernel_name(B, C, Hp, Wp, k, s)
        sub = image_subset(B)
        a_ref, S, floor = dwconv_reference(xp[sub, lo:lo + H, lo:lo + W], a["w"], a["bias"], k, s, lo, hi, ctx["circular"])
        problems = []
        if tuple(a_ref.shape[1:3]) != (Ho, Wo):
            problems.append("output %dx%d, the module's rule gives %dx%d" % (Ho, Wo, a_ref.shape[1], a_ref.shape[2]))
            self._record(entry, kernel, "", [], problems)
            return
        ys = y[sub]
        r = act_check(ys, a_ref, S, floor, TAU["dwconv"])
        ref_s, S_s, floor_s = se_sum_reference(ys, se_sum_conversions(Ho, Wo))
        got_s = sums[sub].to(F64) / cabi.SE_SUM_SCALE
        rs = bound_check(got_s, ref_s, S_s, 0.0, TAU_SUM, floor_s)
        res = [("y", r[0], r[1], "dwconv"), ("y", r[0], r[2], "eps_act"), ("chan_sum",) + rs + ("se_sum",)]
        problems += self._replay(entry, a, "y")
        FEATURES.add(("dw", kernel, k, s))
        if C % 64:
            FEATURES.add(("dw", kernel, k, "C%64"))
        geom = "B%d %dx%d->%dx%d C=%d k%d s%d pad=(%d,%d)%s" % (B, H, W, Ho, Wo, C, k, s, lo, hi,
                                                             " circular" if ctx["circular"] else "")
        self._record(entry, kernel, geom, res, problems)

    def check_se(self, entry, a):
        ctx = self.ctx
        sums, wg, gate_ws, rep = a["chan_sum"], a["wg"], a["gate_ws"], a["rep"]
        w_proj = a["w_proj"]
        cout, mid = w_proj.shape
        B = sums.shape[0]
        hw = ctx.pop("hw")                                   # the depthwise output's Ho * Wo, not the inv_hw argument
        sub = image_subset(B)
        g_ref, wg_ref = se_gate_reference(sums[sub], hw, a["w_red"], a["b_red"], a["w_se"], a["b_se"], w_proj)
        w = wg[sub]
        bound_S = w_proj.to(F64).abs().unsqueeze(0).expand_as(wg_ref)
        res = []
        problems = []
        for r in range(rep):
            for r2 in range(rep):
                blk = w[:, r * cout:(r + 1) * cout, r2 * mid:(r2 + 1) * mid]
                if r == r2:
                    res.append(("wg[%d]" % r,) + bound_check(blk, wg_ref, bound_S, RHO_BF16, TAU_GATE) + ("se_gate",))
                elif not bool((blk == 0).all()):
                    problems.append("off-diagonal block (%d, %d) is not 0" % (r, r2))
        two_launch = gate_ws is not None and not bool(torch.isnan(gate_ws).all())
        if two_launch:
            gate = gate_ws.view(B, mid)[sub]
            res.append(("gate",) + bound_check(gate, g_ref, torch.ones_like(g_ref), 0.0, TAU_GATE) + ("se_gate",))
        kernel = "se_gate_kernel+se_scale_kernel" if two_launch else "se_gate_scale_kernel"
        problems += self._replay(entry, a, "wg")
        ctx["rep"] = rep
        FEATURES.add(("se", kernel, rep))
        self._record(entry, kernel, "B%d mid=%d R=%d cout=%d rep%d hw=%d" % (B, mid, a["w_red"].shape[0], cout, rep, hw),
                     res, problems)

    def check_project(self, entry, a):
        ctx = self.ctx
        i = ctx["block"]
        d, wg, res_t, out, bias, out_b = a["d"], a["wg"], a["residual"], a["out"], a["bias"], a["out_biased"]
        rep = ctx.pop("rep")
        o = ctx["fe"].blocks[i]
        mid, cout = o.mid, o.cout
        B = d.shape[0]
        sub = image_subset(B)
        problems = []
        if (res_t is not None) != bool(ctx["module"]._blocks[i]._residual):
            problems.append("residual given: %s, the module's block has one: %s" % (res_t is not None,
                                                                                    ctx["module"]._blocks[i]._residual))
        ref, S, floor = project_reference(unpack_rep(d[sub], rep, mid), wg[sub][:, :cout, :mid],
                                          None if res_t is None else res_t[sub].reshape(len(sub), -1, cout))
        got = unpack_rep(out[sub], rep, cout)
        res = [("out",) + bound_check(got, ref, S, RHO_BF16, TAU["project"], floor) + ("project",)]
        if out_b is not None:
            if not torch.equal(bias, o.b_proj.repeat(rep)):
                problems.append("the biased copy's bias is not the block's projection bias")
            if not torch.equal(out_b, (out.float() + bias.float()).to(torch.bfloat16)):
                problems.append("out_biased != bf16(out + bias) in %d elements" % int(
                    (out_b != (out.float() + bias.float()).to(torch.bfloat16)).sum()))
            FEATURES.add(("proj", "biased"))
        problems += self._replay(entry, a, "out")
        if res_t is not None:
            FEATURES.add(("proj", "residual"))
        if rep > 1:
            FEATURES.add(("proj", "rep%d" % rep))
        HW = d.numel() // (B * mid)
        geom = "B%d HW=%d mid=%d cout=%d rep%d%s%s" % (B, HW, mid, cout, rep, " +res" if res_t is not None else "",
                                                     " +biased" if out_b is not None else "")
        self._record(entry, "project_tcgen05_kernel", geom, res, problems)

    # -- guarded replay --------------------------------------------------------------------------------------------
    def _replay(self, entry, a, out_name, written=None):
        """Launches the entry once more with every output in a fresh sentinel-guarded buffer (a fresh zeroed chan_sum, a
        fresh NaN gate workspace); returns a list of problems."""
        args = dict(a)
        outs = [out_name] + (["out_biased"] if entry == "mbconv_project_nhwc" and a["out_biased"] is not None else [])
        bufs = {}
        for name in outs:
            t = a[name]
            n = t.numel()
            guard = guard_len(t.shape[-1])
            buf = guarded(n, t.dtype, guard, t.device)
            bufs[name] = (buf, n, guard)
            args[name] = buf[guard:guard + n].view(t.shape)
        if entry == "dwconv_bias_silu_nhwc":
            args["chan_sum"] = torch.zeros_like(a["chan_sum"])
        if entry == "se_gate_scale" and a["gate_ws"] is not None:
            args["gate_ws"] = torch.full_like(a["gate_ws"], float("nan"))
        _ORIG[entry](**args)
        torch.cuda.synchronize()
        problems = []
        for name in outs:
            buf, n, guard = bufs[name]
            problems += ["replay %s: %s" % (name, p) for p in guard_report(buf, n, guard, a[name],
                                                                          written if name == out_name else None)]
        if entry == "dwconv_bias_silu_nhwc" and not torch.equal(args["chan_sum"], a["chan_sum"]):
            problems.append("replay chan_sum differs from the plan's")
        return problems

    # -- report ----------------------------------------------------------------------------------------------------
    def table(self, title, seconds):
        lines = ["", "== %s: %d checked launches, %.1f s ==" % (title, len(self.rows), seconds),
                 "%-22s %-9s %-31s %-52s %10s %10s" % ("entry", "where", "kernel", "geometry", "err/bound", "tau need")]
        for entry, where, kernel, geom, worst, need in self.rows:
            lines.append("%-22s %-9s %-31s %-52s %10.3g %10.3g" % (entry, where, kernel, geom, worst, need))
        return "\n".join(lines)

    def assert_coverage(self):
        for e in ENTRIES:
            if e != "bias_silu_nhwc":
                assert self.checked[e] == self.intercepted[e], (e, self.checked[e], self.intercepted[e])
        assert self.extracts == 2, "%d encoder passes" % self.extracts


# ---------------------------------------------------------------------------------------------------------------
# configurations
# ---------------------------------------------------------------------------------------------------------------
#: name -> (variant, ori_noise, circular, ground shape (H, W), batch, weight seed, uint8 input: None or (shift, crop_w))
CONFIGS = {
    "vigor_b64": ("vigor", None, True, (320, 640), 64, 61, None),
    "kitti_b32": ("kitti", None, None, (256, 1024), 32, 62, None),
    "vigor_prior72_fov180_b64": ("vigor_prior", 72.0, False, (320, 320), 64, 63, None),
    "oxford_b1": ("oxford", None, None, (154, 231), 1, 64, None),
    "vigor_u8_b3": ("vigor", None, True, (320, 640), 3, 65, (False, None)),
    "fov180_u8_b2": ("vigor_prior", 72.0, False, (320, 640), 2, 66, (True, 320)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CONFIGS))
def test_encoder_plan_launches(cuda_device, monkeypatch, name):
    from helpers import build_model
    from ccvpe_b200.synthetic import AERIAL_SHAPE, synthetic_pair
    variant, noise, circular, ghw, batch, wseed, u8 = CONFIGS[name]
    model = build_model(variant, noise, circular, wseed).to(cuda_device).set_precision("bf16").eval()
    model.pipeline.concurrent = False
    t0 = time.time()
    rec = Recorder(monkeypatch, model)
    with torch.no_grad():
        if u8 is None:
            grd, sat = (t.to(cuda_device) for t in synthetic_pair(batch, ghw, seed=wseed))
            out = model(grd, sat)
            assert all(bool(torch.isfinite(t).all()) for t in out)
        else:
            rolled, crop_w = u8
            g = torch.Generator().manual_seed(wseed)
            grd = torch.randint(0, 256, (batch, 3) + ghw, generator=g, dtype=torch.uint8).to(cuda_device)
            sat = torch.randint(0, 256, (batch, 3) + AERIAL_SHAPE, generator=g, dtype=torch.uint8).to(cuda_device)
            shift = torch.randint(-ghw[1], ghw[1], (batch,), generator=g, dtype=torch.int32).to(cuda_device) if rolled else None
            model.localize_u8(grd, sat, shift, crop_w)
    torch.cuda.synchronize()
    print(rec.table(name, time.time() - t0))
    CONFIGS_RUN.add(name)
    assert not rec.failures, "\n".join(rec.failures[:40])
    rec.assert_coverage()


@pytest.mark.gpu
def test_every_encoder_kernel_was_checked(cuda_device):
    """Across the configurations above, every encoder kernel and variant of the plan was reached and checked."""
    if CONFIGS_RUN != set(CONFIGS):
        pytest.skip("needs every configuration of this file in the same run")
    consts = dict(TAU, se_sum=TAU_SUM, se_gate=TAU_GATE, eps_act=EPS_ACT, wrap=0.0)
    print("\nworst tau needed per operator: " + ", ".join("%s %.3g (constant %.0e)" % (k, v, consts[k]) for k, v in
                                                           sorted(MEASURED.items())))
    want = [("stem", "fp32", True), ("stem", "fp32", False), ("stem", "u8", True), ("stem", "u8", False),
            ("dw", "dwconv_bias_silu_kernel", 3, 1), ("dw", "dwconv_bias_silu_kernel", 3, 2),
            ("dw", "dwconv_bias_silu_kernel", 5, 2), ("dw", "dwconv_tile_kernel", 3, 1), ("dw", "dwconv_tile_kernel", 5, 1),
            ("dw", "dwconv_tile_kernel", 3, "C%64"), ("dw", "dwconv_tile_kernel", 5, "C%64"),
            ("se", "se_gate_scale_kernel", 1), ("se", "se_gate_kernel+se_scale_kernel", 1),
            ("se", "se_gate_kernel+se_scale_kernel", 2),
            ("proj", "residual"), ("proj", "biased"), ("proj", "rep2"), ("wrap",)]
    missing = [f for f in want if f not in FEATURES]
    assert not missing, (missing, sorted(FEATURES, key=str))


# ---------------------------------------------------------------------------------------------------------------
# CPU self-test of the checker: the bounds pass a correctly rounded result and fail each planted fault
# ---------------------------------------------------------------------------------------------------------------
def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _bf16(t):
    return t.to(torch.bfloat16)


#: the SiLU approximation error injected into the "correct kernel" outputs below: the measured magnitude, relative to the
#: pre-activation (EPS_ACT is at least 4x this)
EPS_INJECTED = EPS_ACT / 4


def _kernel_act(a, eps=EPS_INJECTED):
    """A correct kernel's activated bf16 output: silu(a) with an approximation error of +-eps |a| (alternating sign),
    rounded once."""
    sign = torch.ones(a.numel(), dtype=a.dtype)
    sign[1::2] = -1
    return _bf16(silu64(a) + eps * a.abs() * sign.view(a.shape))


def _stem_problem(u8):
    g = _gen(31)
    B, H, W = 2, 11, 14
    x = torch.randint(0, 256, (B, 3, H, W), generator=g, dtype=torch.uint8) if u8 else torch.randn(B, 3, H, W, generator=g)
    shift = torch.tensor([5, -9], dtype=torch.int32) if u8 else None
    w = torch.randn(27, 32, generator=g) * 0.3
    bias = torch.randn(32, generator=g) * 0.1
    return x, shift, w, bias


def _dw_problem(C, k, s, circular, seed=32):
    g = _gen(seed)
    B, H, W = 2, 6, 7
    x = _bf16(torch.randn(B, H, W, C, generator=g))
    w = _bf16(torch.randn(k * k, C, generator=g) * 0.4)
    bias = _bf16(torch.randn(C, generator=g) * 0.3)
    lo, hi = ((k - 1) // 2, (k - 1) // 2) if s == 1 else ((k - 2) // 2, k - 2 - (k - 2) // 2)
    return x, w, bias, lo, hi


def _se_problem(rep=1):
    g = _gen(33)
    B, mid, R, cout, hw = 2, 64, 8, 24, 42
    sums = (torch.randn(B, mid, generator=g) * hw * 0.5 * cabi.SE_SUM_SCALE).round().to(torch.int64)
    w_red = _bf16(torch.randn(R, mid, generator=g) / math.sqrt(mid) * 2)
    b_red = _bf16(torch.randn(R, generator=g))
    w_se_t = _bf16(torch.randn(R, mid, generator=g) / math.sqrt(R) * 2)
    b_se = _bf16(torch.randn(mid, generator=g))
    w_proj = _bf16(torch.randn(cout, mid, generator=g))
    return sums, hw, w_red, b_red, w_se_t, b_se, w_proj


def _proj_problem():
    g = _gen(34)
    B, HW, mid, cout = 3, 130, 32, 16                      # 130 pixels: a full and a ragged 128-row tile
    d = _bf16(torch.randn(B, HW, mid, generator=g))
    wg = _bf16(torch.randn(B, cout, mid, generator=g) / math.sqrt(mid))
    res = _bf16(torch.randn(B, HW, cout, generator=g))
    return d, wg, res


def _act_ratio(got, a_ref, S, floor, op):
    return act_check(got, a_ref, S, floor, TAU[op])[0]


def _stem_case(u8, mutate=None):
    x, shift, w, bias = _stem_problem(u8)
    v = stem_operand(x, shift, 12 if u8 else None)
    ref = stem_reference(v, w, bias, 0, 1, u8)
    if mutate == "roll sign":
        v = stem_operand(x, -shift, 12)
    got = _kernel_act(stem_reference(v, w, bias, 0, 1, u8)[0])
    return _act_ratio(got, *ref, "stem")


def _dw_case(C, k, s, circular, mutate=None):
    x, w, bias, lo, hi = _dw_problem(C, k, s, circular)
    ref = dwconv_reference(x, w, bias, k, s, lo, hi, circular)
    b, pl, ph = bias, lo, hi
    xk = x.to(F64).permute(0, 3, 1, 2)
    if mutate == "bias shifted":                           # the last, partial 64-channel block reads bias one channel on
        b = bias.clone()
        b[640:671] = bias[641:672]
    if mutate == "stride-2 pads swapped":
        pl, ph = hi, lo
    if mutate == "border tap reads the interior":          # the left padding column repeats interior column 0
        H = xk.shape[2]
        xpad = F.pad(xk, (lo, hi, lo, hi))
        xpad[:, :, lo:lo + H, 0] = xk[..., 0]
        wk = w.to(F64).t().reshape(C, 1, k, k)
        a = F.conv2d(xpad, wk, bias.to(F64), stride=s, groups=C).permute(0, 2, 3, 1)
        return _act_ratio(_kernel_act(a), *ref, "dwconv")
    if mutate == "wrap column one off":                    # the left wrap column copies interior column W-2, not W-1
        W = xk.shape[3]
        xpad = F.pad(torch.cat([xk[..., W - 2:W - 1], xk, xk[..., :hi]], dim=3), (0, 0, lo, hi))
        wk = w.to(F64).t().reshape(C, 1, k, k)
        a = F.conv2d(xpad, wk, bias.to(F64), stride=s, groups=C).permute(0, 2, 3, 1)
        return _act_ratio(_kernel_act(a), *ref, "dwconv")
    got = _kernel_act(dwconv_reference(x, w, b, k, s, pl, ph, circular)[0])
    return _act_ratio(got, *ref, "dwconv")


def _se_sum_case(mutate=None):
    x, w, bias, lo, hi = _dw_problem(96, 3, 1, False)
    y = _kernel_act(dwconv_reference(x, w, bias, 3, 1, lo, hi, False)[0])
    Ho, Wo = y.shape[1:3]
    ref, S, floor = se_sum_reference(y, se_sum_conversions(Ho, Wo))
    got = ref.clone()
    if mutate == "pixel missing":
        got = got - y[:, 2, 3].to(F64)
    fixed = (got * cabi.SE_SUM_SCALE).round()                 # what the int64 accumulator holds
    return bound_check(fixed / cabi.SE_SUM_SCALE, ref, S, 0.0, TAU_SUM, floor)[0]


def _se_gate_case(mutate=None, rep=1):
    sums, hw, w_red, b_red, w_se_t, b_se, w_proj = _se_problem()
    g_ref, wg_ref = se_gate_reference(sums, hw, w_red, b_red, w_se_t, b_se, w_proj)
    hw_k = 4 * hw if mutate == "inv_hw of the previous block" else hw
    _, wg_k = se_gate_reference(sums, hw_k, w_red, b_red, w_se_t, b_se, w_proj)
    got = _bf16(wg_k)
    return bound_check(got, wg_ref, w_proj.to(F64).abs().unsqueeze(0).expand_as(wg_ref), RHO_BF16, TAU_GATE)[0]


def _proj_case(mutate=None):
    d, wg, res = _proj_problem()
    ref, S, floor = project_reference(d, wg, res)
    B, HW, cout = ref.shape
    if mutate == "packed pixels swapped":                  # rep = 2: two pixels per GEMM row, the halves swapped
        dp, wgp = d.reshape(B, HW // 2, 64), torch.zeros(B, 2 * cout, 64, dtype=torch.bfloat16)
        wgp[:, :cout, :32], wgp[:, cout:, 32:] = wg, wg
        ref, S, floor = project_reference(unpack_rep(dp, 2, 32), wgp[:, :cout, :32], res)
        out = _bf16(project_reference(dp, wgp, res.reshape(B, HW // 2, 2 * cout))[0])
        out = out.view(B, HW // 2, 2, cout).flip(2).reshape(B, HW // 2, 2 * cout)
        return bound_check(unpack_rep(out, 2, cout), ref, S, RHO_BF16, TAU["project"], floor)[0]
    r = res
    if mutate == "residual of image b+1":
        r = res.roll(-1, dims=0)
    out = _bf16(project_reference(d, wg, r)[0])
    if mutate == "last row of a ragged tile zeroed":
        out[:, HW - 1] = 0
    return bound_check(out, ref, S, RHO_BF16, TAU["project"], floor)[0]


def _pw_case(mutate=None):
    g = _gen(35)
    B, H, W, K, N = 2, 5, 7, 40, 48                        # K = 40: a 32-wide block and an 8-channel tail (pad_k_blocks)
    x = _bf16(torch.randn(B, H, W, K, generator=g))
    w_nk = cabi.pad_k_blocks(torch.randn(N, K, generator=g) / math.sqrt(K) * 2)
    bias = torch.randn(N, generator=g) * 0.1
    ref = pointwise_reference(x, w_nk, bias)
    wk = w_nk.clone()
    if mutate == "expand K tail block dropped":
        wk[:, 32:] = 0
    return _act_ratio(_kernel_act(pointwise_reference(x, wk, bias)[0]), *ref, "pointwise")


def test_checker_references_are_the_torch_ops():
    """Each float64 reference is the torch operation it restates, to 1e-12."""
    x, w, bias, lo, hi = _dw_problem(48, 5, 2, False)
    a, S, _ = dwconv_reference(x, w, bias, 5, 2, lo, hi, False)
    xp = F.pad(x.double().permute(0, 3, 1, 2), (lo, hi, lo, hi))
    ref = F.conv2d(xp, w.double().t().reshape(48, 1, 5, 5), bias.double(), stride=2, groups=48).permute(0, 2, 3, 1)
    assert torch.allclose(a, ref, rtol=1e-12, atol=1e-12) and bool((S >= a.abs()).all())
    assert torch.allclose(silu64(a), F.silu(ref), rtol=1e-12, atol=1e-12)
    # circular: the module's own padding (efficientnet.SamePadConv2d)
    from ccvpe_b200.efficientnet import SamePadConv2d
    conv = SamePadConv2d(48, 48, 3, stride=1, groups=48, circular=True).double()
    x, w, bias, lo, hi = _dw_problem(48, 3, 1, True)
    with torch.no_grad():
        conv.weight.copy_(w.double().t().reshape(48, 1, 3, 3))
        ref = conv(x.double().permute(0, 3, 1, 2)).permute(0, 2, 3, 1) + bias.double()
    a, *_ = dwconv_reference(x, w, bias, 3, 1, conv._pad_lo, conv._pad_hi, True)
    assert torch.allclose(a, ref, rtol=1e-12, atol=1e-12)
    stem = SamePadConv2d(3, 32, 3, stride=2, circular=True).double()
    xs, _, ws, bs = _stem_problem(False)
    with torch.no_grad():
        stem.weight.copy_(_bf16(ws).double().t().reshape(32, 3, 3, 3))
        ref = stem(_bf16(xs).double()).permute(0, 2, 3, 1) + bs.double()
    a, *_ = stem_reference(stem_operand(xs), ws, bs, stem._pad_lo, stem._pad_hi, True)
    assert torch.allclose(a, ref, rtol=1e-12, atol=1e-12)
    d, wg, res = _proj_problem()
    ref, S, _ = project_reference(d, wg, res)
    assert torch.allclose(ref, torch.bmm(d.double(), wg.double().transpose(1, 2)) + res.double(), rtol=1e-12, atol=1e-12)
    g = _gen(36)
    xq = _bf16(torch.randn(2, 3, 4, 40, generator=g))
    wq = cabi.pad_k_blocks(torch.randn(24, 40, generator=g))
    bq = torch.randn(24, generator=g)
    a, *_ = pointwise_reference(xq, wq, bq)
    assert torch.allclose(a, F.linear(xq.double(), wq[:, :40].double(), bq.double()), rtol=1e-12, atol=1e-12)


def test_checker_u8_operand_is_the_kernel_fma():
    """bf16(fp32(u8 * sc + sh)) with sc, sh as the kernel's float32 arithmetic: within one fp32 rounding of ToTensor +
    Normalize, and the float64 product + sum is exact (one rounding to fp32 = fmaf)."""
    from fractions import Fraction
    x, shift, _, _ = _stem_problem(True)
    sc, sh = u8_scale_shift(cabi.IMAGENET_MEAN, cabi.IMAGENET_STD)
    for c in range(3):
        for u in range(256):
            f64 = float(u) * float(sc[c]) + float(sh[c])
            assert Fraction(f64) == Fraction(u) * Fraction(float(sc[c])) + Fraction(float(sh[c])), (c, u)
    exact = x.double() * sc.double().view(1, 3, 1, 1) + sh.double().view(1, 3, 1, 1)
    mean = torch.tensor(cabi.IMAGENET_MEAN).view(1, 3, 1, 1).double()
    std = torch.tensor(cabi.IMAGENET_STD, dtype=torch.float32).view(1, 3, 1, 1).double()
    assert (exact - (x.double() / 255 - mean) / std).abs().max() < 1e-5
    v = stem_operand(x, shift, 12)
    assert v.shape[-1] == 12 and torch.equal(v[1, :, :, 0], stem_operand(x)[1, :, :, (0 - int(shift[1])) % x.shape[3]])


def test_checker_passes_a_correct_kernel():
    assert _stem_case(False) <= 1.0 and _stem_case(True) <= 1.0
    for C, k, s, circ in [(672, 5, 1, False), (96, 3, 2, False), (48, 3, 1, True), (144, 5, 2, True)]:
        assert _dw_case(C, k, s, circ) <= 1.0, (C, k, s, circ)
    assert _se_sum_case() <= 1.0
    assert _se_gate_case() <= 1.0
    assert _proj_case() <= 1.0
    assert _pw_case() <= 1.0


_MUTATIONS = {
    "depthwise border tap reads the interior": lambda: _dw_case(96, 3, 1, False, "border tap reads the interior"),
    "circular wrap column one off": lambda: _dw_case(48, 3, 1, True, "wrap column one off"),
    "stride-2 pad_lo / pad_hi swapped": lambda: _dw_case(96, 3, 2, False, "stride-2 pads swapped"),
    "672-channel tail block bias shifted": lambda: _dw_case(672, 5, 1, False, "bias shifted"),
    "pixel missing from an SE channel sum": lambda: _se_sum_case("pixel missing"),
    "inv_hw of the previous block": lambda: _se_gate_case("inv_hw of the previous block"),
    "residual of image b+1": lambda: _proj_case("residual of image b+1"),
    "last row of a ragged projection tile zeroed": lambda: _proj_case("last row of a ragged tile zeroed"),
    "rep 2 packed pixels swapped": lambda: _proj_case("packed pixels swapped"),
    "expand K tail block dropped": lambda: _pw_case("expand K tail block dropped"),
    "u8 roll with the opposite sign": lambda: _stem_case(True, "roll sign"),
}


@pytest.mark.parametrize("mutation", list(_MUTATIONS))
def test_checker_catches(mutation):
    assert _MUTATIONS[mutation]() > 1.0


@pytest.mark.parametrize("op", ["stem", "pointwise", "dwconv"])
def test_checker_catches_a_silu_with_error_2e7(op):
    """A SiLU whose output is off by 2^-7 of its value fails every activated bound."""
    if op == "stem":
        x, shift, w, bias = _stem_problem(False)
        ref = stem_reference(stem_operand(x), w, bias, 0, 1, False)
    elif op == "pointwise":
        g = _gen(37)
        ref = pointwise_reference(_bf16(torch.randn(2, 4, 5, 64, generator=g)),
                                  cabi.pad_k_blocks(torch.randn(32, 64, generator=g) / 4), torch.randn(32, generator=g))
    else:
        x, w, bias, lo, hi = _dw_problem(64, 3, 1, False)
        ref = dwconv_reference(x, w, bias, 3, 1, lo, hi, False)
    got = _bf16(silu64(ref[0]) * (1 + 2.0 ** -7))
    assert _act_ratio(got, *ref, op) > 1.0


def test_replay_report_flags_border_writes():
    """guard_report with a `written` mask: a replay that also wrote a border element, or left an owned one unwritten,
    is reported."""
    out = _bf16(torch.randn(2, 4, 5, 8))
    written = _written_mask(out.shape, 1, 2, 3, False)
    n, guard = out.numel(), 64
    buf = guarded(n, out.dtype, guard, out.device)
    inner = buf[guard:guard + n].view(out.shape)
    inner[written] = out[written]
    assert guard_report(buf, n, guard, out, written) == []
    inner[0, 0, 0, 0] = 0
    assert any("outside" in p for p in guard_report(buf, n, guard, out, written))
    sentinel_bits(inner)[0, 0, 0, 0] = -1
    sentinel_bits(inner)[tuple(written.nonzero()[0].tolist())] = -1
    assert any("unwritten" in p for p in guard_report(buf, n, guard, out, written))
