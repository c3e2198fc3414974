"""Every GEMM / matching launch of the bf16 inference and training plans against a float64 reference of that launch.

The real models run eagerly (`pipeline.concurrent = False`); the plan's entry points are wrapped:

  * `PostEncoderPipeline._igemm`        forward convs, transposed convs, the cell GEMM, the 3x3 data gradients;
  * `PostEncoderTrainer._igemm_strided` the transposed-conv and cell data gradients (channel-slice sources);
  * `PostEncoderTrainer._wgrad`         the weight gradients;
  * `cabi.match_level`, `cabi.match_level_bwd`.

Each wrapper calls the original, synchronises, recomputes the launch in float64 from the operands exactly as stored (bf16
activations, `w_kn` weights, fp32 epilogue vectors) and checks every output element against

    |got - ref| <= rho * |ref| + tau * S (+ a flush-to-zero floor of ~1e-38 per term for the tensor-core GEMMs)

where S is the same operation applied to absolute values (|A||W||row_scale| + |row_r1||r1_w| + |bias| for a GEMM, sum |A||G|
for a weight gradient) and rho = 2^-8 for bf16 stores, 0 for fp32 stores.  A single max-normalised tolerance would let a
dropped K slice or a stale partial tile through: both change a few elements by much less than the tensor's maximum.

The tensor-core GEMM launches are then replayed once into a buffer with sentinel guard bands on both sides and a sentinel-
filled interior: the guards must be intact, no sentinel may remain inside (the plan's launches write every element), and
the interior must be bit-identical to the plan's own output (the tcgen05 igemm, ring and wgrad kernels use no atomics).

The CPU self-test at the end of the file shows that the bound is tight enough to catch the faults it is meant to catch.
"""
import inspect
import time

import pytest
import torch
from torch.nn import functional as F

from ccvpe_b200 import cabi
from ccvpe_b200.decoder import PostEncoderPipeline
from ccvpe_b200.training import PostEncoderTrainer
from oracle import ccvpe_oracle as orc

F64 = torch.float64
RHO_BF16 = 2.0 ** -8

#: tau per operator: at least 4x the worst (|got - ref| - rho |ref| - floor) / S measured on a B200 (1000 W power limit)
#: over every configuration of this file, and never above 1e-4.  Measured worst values:
#:   igemm (tcgen05 generic / halo / ring, every output mode)  5.5e-7  (training VIGOR B=8, level-6 conv_a, K = 9 x 1344)
#:   match_level (tcgen05)                                     1.4e-5  (Oxford level 6: 7-channel windows, norms from prefix sums)
#:   match_level_bwd                                           1.1e-6  (VIGOR B=8, bottleneck level)
#:   wgrad (tcgen05)                                           4.0e-5  (VIGOR B=8, level-1 conv_b: 2.1 million pixels summed in
#:                                                                      fp32, ~u sqrt(M)); capped at 1e-4, a 2.5x margin
TAU = {"igemm": 1e-5, "wgrad": 1e-4, "match": 6e-5, "match_bwd": 1e-5}

#: bf16 launches allowed to resolve to a CUDA-core kernel: {kernel-qualified tag: reason}
SIMT_ALLOWED = {}

SENTINEL = {torch.bfloat16: (torch.int16, -1), torch.float32: (torch.int32, -1)}    # all-ones bits: a NaN no kernel writes


# ---------------------------------------------------------------------------------------------------------------
# float64 references
# ---------------------------------------------------------------------------------------------------------------
def _taps(a, Hout, Wout, stride, k, pad):
    """a [B, Hin, Win, K] (float64) -> list over taps (ty, tx) of [B*Hout*Wout, K]: the input pixel
    (ho*stride - pad + ty, wo*stride - pad + tx) of every output pixel, zero outside the image."""
    B, Hin, Win, K = a.shape
    need_h = (Hout - 1) * stride + k
    need_w = (Wout - 1) * stride + k
    ap = F.pad(a, (0, 0, pad, max(0, need_h - Hin - pad), pad, max(0, need_w - Win - pad)))
    out = []
    for ty in range(k):
        for tx in range(k):
            v = ap[:, ty:ty + (Hout - 1) * stride + 1:stride, tx:tx + (Wout - 1) * stride + 1:stride, :]
            out.append(v.reshape(B * Hout * Wout, K))
    return out


def _operand_a(a0, c0, a1, c1):
    a = a0[..., :c0].to(F64)
    if c1:
        a = torch.cat([a, a1[..., :c1].to(F64)], dim=-1)
    return a


def igemm_reference(a0, c0, a1, c1, geom, w_kn, N, bias=None, row_scale=None, row_r1=None, r1_w=None, relu=False):
    """The implicit GEMM of `ccvpe_igemm` (include/ccvpe_b200.h; igemm_simt.cu is its plain statement) in float64.
    a0 / a1: channels-last [B, Hin, Win, >= c] views as stored; geom = (Hout, Wout, stride, k, pad); w_kn [taps, c0+c1, N];
    row vectors over the B*Hout*Wout output pixels.  Returns (ref, S, floor), all [B*Hout*Wout, N] (see `subnormal_floor`)."""
    Hout, Wout, stride, k, pad = geom
    w = w_kn.to(F64)[:, :, :N]
    y = s = t1 = None
    for t, at in enumerate(_taps(_operand_a(a0, c0, a1, c1), Hout, Wout, stride, k, pad)):
        yt, st, ut = at @ w[t], at.abs() @ w[t].abs(), (at.abs() + 1) @ (w[t].abs() + 1)
        y, s, t1 = (yt, st, ut) if y is None else (y + yt, s + st, t1 + ut)
    floor = subnormal_floor(t1)
    if row_scale is not None:
        rs = row_scale.to(F64).reshape(-1, 1)
        y, s, floor = y * rs, s * rs.abs(), floor * rs.abs().clamp_min(1.0)
    if row_r1 is not None:
        r1, r1w = row_r1.to(F64).reshape(-1, 1), r1_w.to(F64)[:N].reshape(1, -1)
        y, s = y + r1 * r1w, s + (r1 * r1w).abs()
    if bias is not None:
        b = bias.to(F64)[:N].reshape(1, -1)
        y, s = y + b, s + b.abs()
    if relu:
        y = y.clamp_min(0.0)
    return y, s, floor + 4 * TINY                    # (+ the fp32 epilogue's own flushes)


TINY = 2.0 ** -126          # smallest normal fp32 / bf16 magnitude


def subnormal_floor(t1):
    """Absolute allowance for flush-to-zero.  The tensor cores flush subnormal operands, products and partial sums: a term
    a*w of an output loses at most TINY * (|a| + |w| + 2) <= 2 TINY (|a| + 1)(|w| + 1); `t1` is that sum over the output's
    terms.  Without it, gradients that decay into the subnormal range (the orientation loss is a Gaussian blob, so its
    data gradients are ~1e-40 far from the blob) fail the relative bound although they are zero to within 1e-38.  The
    floor stays below 1e-30 for every shape here, far under any value the bound is meant to resolve."""
    return 2 * TINY * t1


def output_as_mn(out, mode, N, ldo, B, Hout, Wout):
    """The kernel's output tensor read back as the [B*Hout*Wout, N] GEMM result (output modes of include/ccvpe_b200.h:
    0 channels-last at row stride ldo; 1 pixel shuffle, n = (2i+j)*cout + co written to (2h+i, 2w+j); 2 planar)."""
    HW = Hout * Wout
    if mode == 0:
        return out.reshape(B, HW, ldo)[:, :, :N].reshape(B * HW, N)
    if mode == 1:
        cout = N // 4
        v = out.reshape(B, Hout, 2, Wout, 2, ldo)[..., :cout]
        return v.permute(0, 1, 3, 2, 4, 5).reshape(B * HW, N)
    return out.reshape(B, N, HW).transpose(1, 2).reshape(B * HW, N)


def mn_as_output(y, mode, N, ldo, B, Hout, Wout):
    """Inverse of `output_as_mn` (the self-test writes its "kernel outputs" with it); ldo == N (or N / 4) only."""
    HW = Hout * Wout
    if mode == 0:
        return y.reshape(B, Hout, Wout, N).contiguous()
    if mode == 1:
        cout = N // 4
        return y.reshape(B, Hout, Wout, 2, 2, cout).permute(0, 1, 3, 2, 4, 5).reshape(B, 2 * Hout, 2 * Wout, cout).contiguous()
    return y.reshape(B, HW, N).transpose(1, 2).reshape(B, N, Hout, Wout).contiguous()


def wgrad_reference(a0, c0, a1, c1, geom, g2d, N, row_scale=None):
    """dW[tap, k, n] = sum_m A[shifted(m, tap), k] * G[m, n] * g_row_scale[m] over all output pixels (`ccvpe_wgrad`);
    geom = (B, Hin, Win, Hout, Wout, stride, k, pad).  Returns (ref, S, floor), all [taps, c0 + c1, N]."""
    B, Hin, Win, Hout, Wout, stride, k, pad = geom
    g = g2d[:, :N].to(F64)
    if row_scale is not None:
        g = g * row_scale.to(F64).reshape(-1, 1)
    taps = _taps(_operand_a(a0, c0, a1, c1), Hout, Wout, stride, k, pad)
    ref = torch.stack([at.t() @ g for at in taps])
    S = torch.stack([at.abs().t() @ g.abs() for at in taps])
    floor = torch.stack([subnormal_floor((at.abs() + 1).t() @ (g.abs() + 1)) for at in taps])
    return ref, S, floor


def _window_index(C, L, base, device):
    return (torch.arange(L, device=device) + base) % C


def match_reference(x, g, offset, shifts, round_g):
    """Scores of one matching level through the oracle (`orc.match_level`, reference models.py:186-202) in float64.
    x [B, C, H, W]; g [B, L] fp32.  The tensor-core kernel correlates with the bf16-rounded descriptor but divides by the
    norm of the fp32 one (`round_g`).  Returns (ref, S) [B, R, H, W]; S = the cosine over absolute values (<= 1)."""
    B, C = x.shape[:2]
    L = g.shape[1]
    centred = offset != 0
    assert not centred or offset == int(C / 2 - L / 2)
    x64, g64 = x.to(F64), g.to(F64)
    gm = g.to(torch.bfloat16).to(F64) if round_g else g64
    ref = orc.match_level(x64, gm, shifts, 1, centred)
    S = orc.match_level(x64.abs(), gm.abs(), shifts, 1, centred)
    if round_g:
        f = (gm.norm(dim=1) / g64.norm(dim=1)).view(B, 1, 1, 1)
        ref, S = ref * f, S * f
    return ref, S


def match_bwd_reference(x, g, offset, shifts, mask, scores, ds, dscl, dmax, dxh):
    """The backward of one matching level as `ccvpe_match_level_bwd` defines it (train_ops.cu), in float64, from the SAVED
    forward scores (they pick the argmax and enter the normalisation term):
        dS_i = ds_i + dscl_i + [i == first argmax over the masked rolls] * dmax
        dx   = (dxh - xhat <xhat, dxh>) / |x| + sum_i dS_i (G_i / (n_i |g|) - s_i M_i x / n_i^2)
        dg_k = sum_p sum_i dS_i (x[(k + base_i) % C] / (n_i |g|) - s_i g_k / |g|^2)
    x [B, P, C]; g [B, L]; scores / ds [B, R, P]; dscl [B, P, R]; dmax [B, P]; dxh [B, P, C] (the summed contributions);
    any gradient may be None.  Returns (dx, S_dx, dg, S_dg)."""
    B, P, C = x.shape
    L = g.shape[1]
    R = len(shifts)
    dev = x.device
    x, g, s = x.to(F64), g.to(F64), scores.to(F64)
    gn = g.norm(dim=1).view(B, 1)
    dS = torch.zeros(B, R, P, dtype=F64, device=dev)
    if ds is not None:
        dS += ds.to(F64)
    if dscl is not None:
        dS += dscl.to(F64).transpose(1, 2)
    if dmax is not None:
        sel = [i for i in range(R) if (mask >> i) & 1]
        arg = torch.tensor(sel, device=dev)[s[:, sel].argmax(dim=1)]                      # [B, P], first maximum
        dS.scatter_add_(1, arg.unsqueeze(1), dmax.to(F64).unsqueeze(1))
    dx = torch.zeros(B, P, C, dtype=F64, device=dev)
    Sdx = torch.zeros_like(dx)
    dg = torch.zeros(B, L, dtype=F64, device=dev)
    Sdg = torch.zeros_like(dg)
    csum = torch.zeros(B, dtype=F64, device=dev)
    cabs = torch.zeros(B, dtype=F64, device=dev)
    for i, sh in enumerate(shifts):
        idx = _window_index(C, L, offset + sh, dev)
        n2 = x[:, :, idx].pow(2).sum(dim=2)                                               # [B, P]
        n = n2.sqrt()
        co = torch.where(dS[:, i] == 0, torch.zeros_like(n), dS[:, i] / (n * gn))
        be = torch.where(dS[:, i] == 0, torch.zeros_like(n), dS[:, i] * s[:, i] / n2)
        xi = x[:, :, idx]
        dx[:, :, idx] += co.unsqueeze(2) * g.unsqueeze(1) - be.unsqueeze(2) * xi
        Sdx[:, :, idx] += co.abs().unsqueeze(2) * g.abs().unsqueeze(1) + be.abs().unsqueeze(2) * xi.abs()
        dg += torch.einsum("bp,bpk->bk", co, xi)
        Sdg += torch.einsum("bp,bpk->bk", co.abs(), xi.abs())
        csum += (dS[:, i] * s[:, i]).sum(dim=1)
        cabs += (dS[:, i] * s[:, i]).abs().sum(dim=1)
    dg -= g * (csum.view(B, 1) / gn.pow(2))
    Sdg += g.abs() * (cabs.view(B, 1) / gn.pow(2))
    if dxh is not None:
        d = dxh.to(F64)
        nrm = x.norm(dim=2, keepdim=True).clamp_min(1e-12)
        xh = x / nrm
        dx += (d - xh * (xh * d).sum(dim=2, keepdim=True)) / nrm
        Sdx += (d.abs() + xh.abs() * (xh * d).abs().sum(dim=2, keepdim=True)) / nrm
    return dx, Sdx, dg, Sdg


def bound_check(got, ref, S, rho, tau, floor=0.0):
    """Returns (worst |got - ref| / (rho |ref| + tau S + floor), worst (|got - ref| - rho |ref| - floor) / S = the tau this
    tensor needs).  Where the bound is zero the element must be exact; a non-finite output where the reference is finite
    fails."""
    got, ref, S = got.to(F64).reshape(-1), ref.to(F64).reshape(-1), S.to(F64).reshape(-1)
    if torch.is_tensor(floor):
        floor = floor.to(F64).reshape(-1)
    d = (got - ref).abs()
    d = torch.where(torch.isfinite(d), d, torch.full_like(d, float("inf")))
    bound = rho * ref.abs() + tau * S + floor
    ratio = torch.where(bound > 0, d / bound.clamp_min(1e-300), torch.where(d > 0, float("inf"), 0.0))
    excess = (d - rho * ref.abs() - floor).clamp_min(0.0)
    need = torch.where(S > 0, excess / S.clamp_min(1e-300), torch.where(excess > 0, float("inf"), 0.0))
    return (float(ratio.max()) if ratio.numel() else 0.0), (float(need.max()) if need.numel() else 0.0)


def _rho(t):
    return RHO_BF16 if t.dtype == torch.bfloat16 else 0.0


def image_subset(B):
    """Images whose outputs are checked for the per-image operators: all of them up to 8, else 0, 1, B/2 and B-1."""
    return list(range(B)) if B <= 8 else sorted({0, 1, B // 2, B - 1})


# ---------------------------------------------------------------------------------------------------------------
# guarded replay
# ---------------------------------------------------------------------------------------------------------------
def _bits(t):
    ity, _ = SENTINEL[t.dtype]
    return t.view(ity)


def _guarded(n, dtype, guard, dev):
    buf = torch.empty(guard + n + guard, dtype=dtype, device=dev)
    _bits(buf).fill_(SENTINEL[dtype][1])
    return buf


def _guard_report(buf, n, guard, ref_out):
    s = SENTINEL[buf.dtype][1]
    bits = _bits(buf)
    problems = []
    if not bool((bits[:guard] == s).all()):
        problems.append("wrote %d elements before the output" % int((bits[:guard] != s).sum()))
    if not bool((bits[guard + n:] == s).all()):
        problems.append("wrote %d elements past the output" % int((bits[guard + n:] != s).sum()))
    inner = bits[guard:guard + n]
    if bool((inner == s).any()):
        problems.append("left %d output elements unwritten" % int((inner == s).sum()))
    if not torch.equal(inner, _bits(ref_out.reshape(-1))):
        problems.append("replay differs from the plan's output in %d elements" % int((inner != _bits(ref_out.reshape(-1))).sum()))
    return problems


def _guard_len(row):
    return (128 * row + 4096 + 511) // 512 * 512          # >= one 128-row tile; keeps the interior 1 KB aligned


def replay_igemm(d, out):
    """Launches the plan's descriptor once more into a sentinel-guarded buffer; returns a list of problems."""
    n = out.numel()
    guard = _guard_len(max(d.N, d.ldo))
    buf = _guarded(n, out.dtype, guard, out.device)
    d2 = cabi.IgemmDesc.from_buffer_copy(d)
    d2.out = buf[guard:].data_ptr()
    _ORIG["cabi.igemm"](d2)
    torch.cuda.synchronize()
    return _guard_report(buf, n, guard, out)


def replay_wgrad(d, out):
    n = out.numel()
    guard = _guard_len(d.N)
    buf = _guarded(n, out.dtype, guard, out.device)
    d2 = cabi.WgradDesc.from_buffer_copy(d)
    n_ws = cabi.wgrad_workspace_elems(d2)
    ws = torch.empty(n_ws, dtype=torch.float32, device=out.device)
    d2.workspace, d2.workspace_elems = ws.data_ptr(), n_ws
    d2.out = buf[guard:].data_ptr()
    _ORIG["cabi.wgrad"](d2)
    torch.cuda.synchronize()
    return _guard_report(buf, n, guard, out)


# ---------------------------------------------------------------------------------------------------------------
# the recorder
# ---------------------------------------------------------------------------------------------------------------
_ORIG = {"cabi.igemm": cabi.igemm, "cabi.wgrad": cabi.wgrad}
KERNELS_SEEN = set()
CONFIGS_RUN = set()
MEASURED = {}                 # operator -> worst tau needed over the file


class Recorder:
    ENTRIES = ("_igemm", "_igemm_strided", "_wgrad", "match_level", "match_level_bwd")

    def __init__(self, monkeypatch):
        self.rows = []            # (entry, tag, kernel, geometry, worst err/bound, tau needed)
        self.failures = []
        self.intercepted = dict.fromkeys(self.ENTRIES, 0)
        self.checked = dict.fromkeys(self.ENTRIES, 0)
        self.descs = []
        self._install(monkeypatch)

    # -- bookkeeping ---------------------------------------------------------------------------------------------
    def _record(self, entry, tag, kernel, geom, results, problems=()):
        """results: list of (name, ratio, need, operator)"""
        worst = max(r[1] for r in results)
        need = max(r[2] for r in results)
        for name, ratio, nd, op in results:
            MEASURED[op] = max(MEASURED.get(op, 0.0), nd)
            if not ratio <= 1.0:
                self.failures.append("%s %s [%s, %s] %s: err/bound %.3g (tau would need %.3g)" % (entry, tag, kernel, geom,
                                                                                                     name, ratio, nd))
        for p in problems:
            self.failures.append("%s %s [%s, %s] guarded replay: %s" % (entry, tag, kernel, geom, p))
        KERNELS_SEEN.add(kernel)
        self.rows.append((entry, tag, kernel, geom, worst, need))
        self.checked[entry] += 1

    def _check_simt(self, entry, tag, kernel, dtype):
        if dtype == torch.bfloat16 and kernel.endswith("simt_kernel") and (kernel + ":" + tag) not in SIMT_ALLOWED:
            self.failures.append("%s %s resolved to the CUDA-core kernel %s" % (entry, tag, kernel))

    # -- wrappers --------------------------------------------------------------------------------------------------
    def _install(self, mp):
        rec = self

        def igemm_spy(d):
            rec.descs.append(cabi.IgemmDesc.from_buffer_copy(d))
            _ORIG["cabi.igemm"](d)

        def wgrad_spy(d):
            rec.descs.append(cabi.WgradDesc.from_buffer_copy(d))
            _ORIG["cabi.wgrad"](d)

        mp.setattr(cabi, "igemm", igemm_spy)
        mp.setattr(cabi, "wgrad", wgrad_spy)

        def wrap_method(cls, name, check):
            orig = getattr(cls, name)
            sig = inspect.signature(orig)

            def wrapper(self, *args, **kwargs):
                rec.intercepted[name] += 1
                n0 = len(rec.descs)
                res = orig(self, *args, **kwargs)
                torch.cuda.synchronize()
                assert len(rec.descs) == n0 + 1, "%s launched %d GEMMs" % (name, len(rec.descs) - n0)
                ba = sig.bind(self, *args, **kwargs)
                ba.apply_defaults()
                check(ba.arguments, rec.descs[-1], res)
                return res

            mp.setattr(cls, name, wrapper)

        wrap_method(PostEncoderPipeline, "_igemm", lambda a, d, res: rec.check_igemm("_igemm", a, d))
        wrap_method(PostEncoderTrainer, "_igemm_strided", lambda a, d, res: rec.check_igemm("_igemm_strided", a, d))
        wrap_method(PostEncoderTrainer, "_wgrad", lambda a, d, res: rec.check_wgrad(a, d, res))

        orig_ml, orig_mlb = cabi.match_level, cabi.match_level_bwd
        sig_ml, sig_mlb = inspect.signature(orig_ml), inspect.signature(orig_mlb)

        def match_level(*args, **kwargs):
            rec.intercepted["match_level"] += 1
            orig_ml(*args, **kwargs)
            torch.cuda.synchronize()
            ba = sig_ml.bind(*args, **kwargs)
            ba.apply_defaults()
            rec.check_match(ba.arguments)

        def match_level_bwd(*args, **kwargs):
            rec.intercepted["match_level_bwd"] += 1
            orig_mlb(*args, **kwargs)
            torch.cuda.synchronize()
            rec.check_match_bwd(sig_mlb.bind(*args, **kwargs).arguments)

        mp.setattr(cabi, "match_level", match_level)
        mp.setattr(cabi, "match_level_bwd", match_level_bwd)

    # -- checks ----------------------------------------------------------------------------------------------------
    def check_igemm(self, entry, a, d):
        tag = a["tag"]
        a0, c0, B = a["a0"], a["c0"], a["B"]
        a1, c1 = a.get("a1"), a.get("c1", 0)
        Hout, Wout, N, out, mode = a["Hout"], a["Wout"], a["N"], a["out"], a["out_mode"]
        ldo = a["ldo"] if a["ldo"] is not None else N
        wt = a["wt"]
        kernel = cabi.igemm_kernel_name(d)
        self._check_simt(entry, tag, kernel, a["dtype"])
        geom = "B%d %dx%d->%dx%d k%d s%d K=%d+%d N=%d mode%d ldo=%d ld0=%d" % (B, a["Hin"], a["Win"], Hout, Wout, a["k"],
                                                                              a["stride"], c0, c1, N, mode, ldo, d.ld0)
        # the descriptor the library saw describes the tensors in hand
        assert d.a0 == a0.data_ptr() and d.ld0 == a0.stride(-2) and d.c0 == c0 and d.N == N and d.out == out.data_ptr(), geom
        sub = image_subset(B)
        per_img = lambda t: None if t is None else t.reshape(B, -1)[sub].reshape(-1)
        ref, S, floor = igemm_reference(a0[sub], c0, a1[sub] if a1 is not None else None, c1,
                                 (Hout, Wout, a["stride"], a["k"], a["pad"]), wt["w_kn"], N, bias=wt.get("bias"),
                                 row_scale=per_img(a.get("row_scale")), row_r1=per_img(a.get("row_r1")),
                                 r1_w=a.get("r1_w"), relu=bool(a.get("relu")))
        got = output_as_mn(out[sub], mode, N, ldo, len(sub), Hout, Wout)
        ratio, need = bound_check(got, ref, S, _rho(out), TAU["igemm"], floor)
        problems = []
        if kernel != "igemm_simt_kernel":
            assert out.numel() == B * Hout * Wout * N, "the plan's launches write every element of their output"
            problems = replay_igemm(d, out)
        self._record(entry, tag, kernel, geom, [("out", ratio, need, "igemm")], problems)

    def check_wgrad(self, a, d, out):
        tag = a["tag"]
        geom_t = a["geom"]
        a0, c0, a1, c1, g2d, N = a["a0"], a["c0"], a["a1"], a["c1"], a["g2d"], a["N"]
        kernel = cabi.wgrad_kernel_name(d)
        self._check_simt("_wgrad", tag, kernel, a["dtype"])
        B, Hin, Win, Hout, Wout, stride, k, pad = geom_t
        geom = "B%d %dx%d->%dx%d k%d s%d K=%d+%d N=%d ld0=%d ldg=%d" % (B, Hin, Win, Hout, Wout, k, stride, c0, c1, N, d.ld0,
                                                                       d.ldg)
        assert d.a0 == a0.data_ptr() and d.ld0 == a0.stride(-2) and d.g == g2d.data_ptr() and d.ldg == g2d.stride(-2), geom
        ref, S, floor = wgrad_reference(a0, c0, a1, c1, geom_t, g2d, N, a["row_scale"])
        ratio, need = bound_check(out.reshape(ref.shape), ref, S, 0.0, TAU["wgrad"], floor)
        problems = replay_wgrad(d, out) if kernel != "wgrad_simt_kernel" else []
        self._record("_wgrad", tag, kernel, geom, [("dW", ratio, need, "wgrad")], problems)

    def check_match(self, a):
        x, g, offset, shifts, mask = a["x"], a["g"], a["offset"], list(a["shifts"]), a["max_mask"]
        B, H, W, C = x.shape
        L, R = g.shape[1], len(shifts)
        ld_cl = 0 if a["scores_cl"] is None else a["scores_cl"].shape[-1]
        kernel = cabi.match_kernel_name(x.dtype, C, L, offset, shifts, ld_cl, a["backend"])
        geom = "B%d %dx%d C=%d L=%d R=%d off=%d" % (B, H, W, C, L, R, offset)
        tag = "match|C%d" % C
        sub = image_subset(B)
        xs = x[sub].permute(0, 3, 1, 2)
        ref, S = match_reference(xs, g[sub], offset, shifts, round_g=kernel == "match_tcgen05_kernel")
        tau = TAU["match"]
        res = []
        if a["scores"] is not None:
            res.append(("scores",) + bound_check(a["scores"][sub], ref, S, 0.0, tau) + ("match",))
        sel = [i for i in range(R) if (mask >> i) & 1]
        if a["max_out"] is not None:
            res.append(("max",) + bound_check(a["max_out"][sub], ref[:, sel].max(dim=1)[0], S[:, sel].max(dim=1)[0], 0.0, tau)
                       + ("match",))
        nrm = xs.to(F64).norm(dim=1)
        if a["inv_norm"] is not None:
            inv = 1.0 / nrm.clamp_min(1e-12)
            res.append(("inv_norm",) + bound_check(a["inv_norm"][sub], inv, inv, 0.0, tau) + ("match",))
        if a["xhat"] is not None:
            xh = (xs.to(F64) / nrm.clamp_min(1e-12).unsqueeze(1)).permute(0, 2, 3, 1)
            res.append(("xhat",) + bound_check(a["xhat"][sub], xh, xh.abs(), RHO_BF16, tau) + ("match",))
        if a["scores_cl"] is not None:
            cl = a["scores_cl"][sub]
            zero = torch.zeros(cl.shape[:-1] + (ld_cl - R,), dtype=F64, device=cl.device)
            res.append(("scores_cl",) + bound_check(cl, torch.cat([ref.permute(0, 2, 3, 1), zero], dim=-1),
                                                    torch.cat([S.permute(0, 2, 3, 1), zero], dim=-1), _rho(cl), tau)
                       + ("match",))
        self._record("match_level", tag, kernel, geom, res)

    def check_match_bwd(self, a):
        x, g, offset, shifts, mask, scores = a["x"], a["g"], a["offset"], list(a["shifts"]), a["max_mask"], a["scores"]
        B, H, W, C = x.shape
        L, R, P = g.shape[1], len(shifts), H * W
        geom = "B%d %dx%d C=%d L=%d R=%d off=%d" % (B, H, W, C, L, R, offset)
        sub = image_subset(B)
        two_d =lambda t, n: None if t is None else torch.stack([t[b * P:(b + 1) * P, :n] for b in sub])
        dxh = two_d(a["d_xhat"], C)
        if a["d_xhat2"] is not None:
            dxh = dxh.to(F64) + two_d(a["d_xhat2"], C).to(F64)
        dmax = two_d(a["d_max"], 1)
        dx_ref, Sdx, dg_ref, Sdg = match_bwd_reference(
            x[sub].reshape(len(sub), P, C), g[sub], offset, shifts, mask, scores[sub].reshape(len(sub), R, P),
            None if a["d_scores"] is None else a["d_scores"][sub].reshape(len(sub), R, P),
            two_d(a["d_scores_cl"], R), None if dmax is None else dmax[..., 0], dxh)
        tau = TAU["match_bwd"]
        dx = a["dx"][sub].reshape(len(sub), P, C)
        res = [("dx",) + bound_check(dx, dx_ref, Sdx, _rho(dx), tau) + ("match_bwd",),
               ("dg",) + bound_check(a["dg"][sub], dg_ref, Sdg, 0.0, tau) + ("match_bwd",)]
        self._record("match_level_bwd", "match_bwd|C%d" % C, "match_level_bwd_kernel", geom, res)

    # -- report ----------------------------------------------------------------------------------------------------
    def table(self, title, seconds):
        lines = ["", "== %s: %d checked launches, %.1f s ==" % (title, len(self.rows), seconds),
                 "%-16s %-26s %-26s %-62s %10s %10s" % ("entry", "tag", "kernel", "geometry", "err/bound", "tau need")]
        for entry, tag, kernel, geom, worst, need in self.rows:
            lines.append("%-16s %-26s %-26s %-62s %10.3g %10.3g" % (entry, tag, kernel, geom, worst, need))
        return "\n".join(lines)

    def assert_coverage(self, entries):
        for e in self.ENTRIES:
            assert self.checked[e] == self.intercepted[e], (e, self.checked[e], self.intercepted[e])
        for e in entries:
            assert self.checked[e] > 0, "no %s launch was checked" % e


# ---------------------------------------------------------------------------------------------------------------
# configurations
# ---------------------------------------------------------------------------------------------------------------
#: name -> (variant, ori_noise, circular, ground shape key, batch, weight seed)
INFERENCE = {
    "vigor_b64": ("vigor", None, True, "vigor", 64, 51),
    "kitti_b32": ("kitti", None, None, "kitti", 32, 52),
    "vigor_prior72_fov180_b64": ("vigor_prior", 72.0, False, "vigor_fov180", 64, 53),
    "oxford_b1": ("oxford", None, None, "oxford", 1, 54),
    "vigor_b3": ("vigor", None, True, "vigor", 3, 55),
}
TRAINING = {
    "train_vigor_b8": ("vigor", None, True, "vigor", 8, 56, 20),
    "train_kitti_b1": ("kitti", None, None, "kitti", 1, 57, 16),
    "train_oxford_b1": ("oxford", None, None, "oxford", 1, 58, 20),
}


def _model(variant, noise, circular, wseed, dev):
    from helpers import build_model
    m = build_model(variant, noise, circular, wseed).to(dev).set_precision("bf16").eval()
    m.pipeline.concurrent = False
    return m


def _finish(rec, name, t0, entries):
    dt = time.time() - t0
    print(rec.table(name, dt))
    CONFIGS_RUN.add(name)
    assert not rec.failures, "\n".join(rec.failures[:40])
    rec.assert_coverage(entries)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(INFERENCE))
def test_inference_plan_launches(cuda_device, monkeypatch, name):
    from ccvpe_b200.synthetic import GROUND_SHAPES, synthetic_pair
    variant, noise, circular, shape_key, batch, wseed = INFERENCE[name]
    model = _model(variant, noise, circular, wseed, cuda_device)
    grd, sat = (t.to(cuda_device) for t in synthetic_pair(batch, GROUND_SHAPES[shape_key], seed=wseed))
    t0 = time.time()
    rec = Recorder(monkeypatch)
    with torch.no_grad():
        out = model(grd, sat)
    torch.cuda.synchronize()
    assert all(bool(torch.isfinite(t).all()) for t in out)
    _finish(rec, name, t0, ("_igemm", "match_level"))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(TRAINING))
def test_training_plan_launches(cuda_device, monkeypatch, name):
    from ccvpe_b200 import losses
    from ccvpe_b200.synthetic import GROUND_SHAPES, synthetic_ground_truth, synthetic_pair
    variant, noise, circular, shape_key, batch, wseed, n_bins = TRAINING[name]
    model = _model(variant, noise, circular, wseed, cuda_device)
    for p_ in model.parameters():
        p_.requires_grad_(True)
    grd, sat = (t.to(cuda_device) for t in synthetic_pair(batch, GROUND_SHAPES[shape_key], seed=wseed))
    gts = [t.to(cuda_device) for t in synthetic_ground_truth(batch, seed=wseed, n_bins=n_bins)]
    t0 = time.time()
    rec = Recorder(monkeypatch)
    loss = losses.training_loss(model(grd, sat), *gts)
    loss.backward()
    torch.cuda.synchronize()
    assert torch.isfinite(loss)
    _finish(rec, name, t0, Recorder.ENTRIES)


@pytest.mark.gpu
def test_every_tensor_core_kernel_was_checked(cuda_device):
    """Across the configurations above, every tensor-core kernel of the plans was reached and checked."""
    if CONFIGS_RUN != set(INFERENCE) | set(TRAINING):
        pytest.skip("needs every configuration of this file in the same run")
    print("\nworst tau needed per operator: " + ", ".join("%s %.3g (tau %.0e)" % (k, v, TAU[k]) for k, v in
                                                           sorted(MEASURED.items())))
    for k in ("igemm_tcgen05_kernel", "conv_ring_tcgen05_kernel", "wgrad_tcgen05_kernel", "match_tcgen05_kernel"):
        assert k in KERNELS_SEEN, (k, sorted(KERNELS_SEEN))


# ---------------------------------------------------------------------------------------------------------------
# CPU self-test of the checker: the bound passes a correctly rounded result and fails each planted fault
# ---------------------------------------------------------------------------------------------------------------
def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _bf16(t):
    return t.to(torch.bfloat16)


def _conv_problem():
    """3x3 pad-1 conv over two sources, M = 3*8*8 = 192 (a full and a partial 128-row tile), N = 40 (three 16-wide tiles),
    row scale, bias, ReLU: the operands as the plan stores them."""
    g = _gen(7)
    B, H, W, c0, c1, N = 3, 8, 8, 24, 16, 40
    a0 = _bf16(torch.randn(B, H, W, c0, generator=g))
    a1 = _bf16(torch.randn(B, H, W, c1, generator=g))
    w_kn = _bf16(torch.randn(9, c0 + c1, N, generator=g) / (9 * (c0 + c1)) ** 0.5)
    bias = torch.randn(N, generator=g)
    rs = torch.rand(B * H * W, generator=g) * 1.5 + 0.5
    return dict(a0=a0, c0=c0, a1=a1, c1=c1, geom=(H, W, 1, 3, 1), w_kn=w_kn, N=N, bias=bias, row_scale=rs, relu=True), (B, H, W)


def _deconv_problem():
    """k2 s2 transposed conv as a 1x1 GEMM with pixel-shuffle output (N = 4 * 16), row scale + rank-1 + bias."""
    g = _gen(8)
    B, H, W, C, cout = 2, 4, 4, 48, 16
    a0 = _bf16(torch.randn(B, H, W, C, generator=g))
    w_kn = _bf16(torch.randn(1, C, 4 * cout, generator=g) / C ** 0.5)
    return dict(a0=a0, c0=C, a1=None, c1=0, geom=(H, W, 1, 1, 0), w_kn=w_kn, N=4 * cout,
                bias=torch.randn(cout, generator=g).repeat(4), row_scale=torch.rand(B * H * W, generator=g) * 0.5 + 1.25,
                row_r1=torch.randn(B * H * W, generator=g), r1_w=torch.randn(4 * cout, generator=g)), (B, H, W)


def _kernel_output(p, mode, shape, **override):
    """A correct kernel's bf16 output: the float64 result rounded once, written in output mode `mode`."""
    q = dict(p, **override)
    y, *_ = igemm_reference(**q)
    B, H, W = shape
    return mn_as_output(_bf16(y), mode, p["N"], p["N"] if mode == 0 else p["N"] // 4, B, H, W)


def _ratio(p, mode, shape, out):
    ref, S, floor = igemm_reference(**p)
    B, H, W = shape
    got = output_as_mn(out, mode, p["N"], p["N"] if mode == 0 else p["N"] // 4, B, H, W)
    return bound_check(got, ref, S, RHO_BF16, TAU["igemm"], floor)[0]


def test_checker_igemm_reference_is_the_convolution():
    """The float64 reference is the convolution torch computes (3x3 two-source conv and the k2 s2 transposed conv)."""
    p, (B, H, W) = _conv_problem()
    y, *_ = igemm_reference(**dict(p, row_scale=None, relu=False))
    x = torch.cat([p["a0"], p["a1"]], dim=-1).double().permute(0, 3, 1, 2)
    w = p["w_kn"].double().view(3, 3, p["c0"] + p["c1"], p["N"]).permute(3, 2, 0, 1)
    ref = F.conv2d(x, w, p["bias"].double(), padding=1).permute(0, 2, 3, 1).reshape(-1, p["N"])
    assert torch.allclose(y, ref, rtol=1e-12, atol=1e-12)
    q, (B, H, W) = _deconv_problem()
    y, *_ = igemm_reference(**dict(q, row_scale=None, row_r1=None))
    cout = q["N"] // 4
    wt = q["w_kn"][0].double().view(q["c0"], 2, 2, cout).permute(0, 3, 1, 2)
    ref = F.conv_transpose2d(q["a0"].double().permute(0, 3, 1, 2), wt, q["bias"][:cout].double(), stride=2)
    got = mn_as_output(y, 1, q["N"], cout, B, H, W)
    assert torch.allclose(got.permute(0, 3, 1, 2), ref, rtol=1e-12, atol=1e-12)


def test_checker_passes_a_correct_kernel():
    p, shape = _conv_problem()
    assert _ratio(p, 0, shape, _kernel_output(p, 0, shape)) <= 1.0
    q, shape_q = _deconv_problem()
    assert _ratio(q, 1, shape_q, _kernel_output(q, 1, shape_q)) <= 1.0
    assert _ratio(q, 2, shape_q, _kernel_output(q, 2, shape_q)) <= 1.0


def _mutations():
    p, shape = _conv_problem()
    q, shape_q = _deconv_problem()
    B, H, W = shape
    out = {}
    w = p["w_kn"].clone()
    w[4, 16:32] = 0                                                            # centre tap, channels 16..31
    out["K slice of one tap dropped"] = (p, 0, shape, _kernel_output(p, 0, shape, w_kn=w))
    b = p["bias"].clone()
    b[16:32] = p["bias"][17:33]                                                # second 16-wide N tile reads one column on
    out["bias of one N tile shifted"] = (p, 0, shape, _kernel_output(p, 0, shape, bias=b))
    o = _kernel_output(p, 0, shape)
    o.view(-1, p["N"])[B * H * W - 1] = 0                                      # last row of the partial second M tile
    out["last row of a partial M tile zeroed"] = (p, 0, shape, o)
    o = _kernel_output(q, 1, shape_q)
    Bq, Hq, Wq = shape_q
    o = o.view(Bq, Hq, 2, Wq, 2, -1).transpose(2, 4).reshape(o.shape).contiguous()
    out["pixel shuffle (i, j) swapped"] = (q, 1, shape_q, o)
    rs = q["row_scale"].clone()
    rs[5] = 1.0
    out["row_scale missing at one pixel"] = (q, 1, shape_q, _kernel_output(q, 1, shape_q, row_scale=rs))
    # right border: tap column 2 of the last output column reads input column W-1 instead of the zero padding
    y, *_ = igemm_reference(**p)
    a = torch.cat([p["a0"], p["a1"]], dim=-1).double()
    extra = torch.zeros(B, H, W, p["N"], dtype=F64)
    for ty in range(3):
        for h in range(H):
            hi = h + ty - 1
            if 0 <= hi < H:
                extra[:, h, W - 1] += a[:, hi, W - 1] @ p["w_kn"][ty * 3 + 2].double()
    yb, *_ = igemm_reference(**dict(p, relu=False))
    yb = yb + extra.reshape(-1, p["N"]) * p["row_scale"].double().view(-1, 1)
    out["border tap read one column off"] = (p, 0, shape, mn_as_output(_bf16(yb.clamp_min(0)), 0, p["N"], p["N"], B, H, W))
    o = _kernel_output(p, 0, shape).double()
    i = int(y.abs().argmax())
    o.view(-1)[i] = y.view(-1)[i] * 1.02
    out["largest element moved by 2 %"] = (p, 0, shape, o)
    return out


_MUTATION_NAMES = ["K slice of one tap dropped", "bias of one N tile shifted", "last row of a partial M tile zeroed",
                   "pixel shuffle (i, j) swapped", "row_scale missing at one pixel", "border tap read one column off",
                   "largest element moved by 2 %"]


@pytest.mark.parametrize("mutation", _MUTATION_NAMES)
def test_checker_catches(mutation):
    p, mode, shape, out = _mutations()[mutation]
    assert _ratio(p, mode, shape, out) > 1.0


def test_checker_wgrad_reference_is_autograd():
    g = _gen(9)
    B, H, W, c0, c1, N = 2, 6, 8, 16, 8, 24
    x0 = _bf16(torch.randn(B, H, W, c0, generator=g))
    x1 = _bf16(torch.randn(B, H, W, c1, generator=g))
    dy = torch.randn(B, H, W, N, generator=g)
    ref, S, _ = wgrad_reference(x0, c0, x1, c1, (B, H, W, H, W, 1, 3, 1), dy.reshape(-1, N), N)
    w = torch.zeros(N, c0 + c1, 3, 3, dtype=F64, requires_grad=True)
    x = torch.cat([x0, x1], dim=-1).double().permute(0, 3, 1, 2)
    (F.conv2d(x, w, padding=1) * dy.double().permute(0, 3, 1, 2)).sum().backward()
    assert torch.allclose(ref.view(3, 3, c0 + c1, N).permute(3, 2, 0, 1), w.grad, rtol=1e-12, atol=1e-12)
    assert bool((S >= ref.abs()).all())
    # k2 s2 (transposed-conv weight gradient): A = dY at twice the resolution, G = the layer input, row scale on G
    dY = _bf16(torch.randn(B, 2 * H, 2 * W, c0, generator=g))
    xin = _bf16(torch.randn(B, H, W, N, generator=g))
    rs = torch.rand(B * H * W, generator=g) + 0.5
    ref, *_ = wgrad_reference(dY, c0, None, 0, (B, 2 * H, 2 * W, H, W, 2, 2, 0), xin.reshape(-1, N), N, rs)
    w = torch.zeros(N, c0, 2, 2, dtype=F64, requires_grad=True)
    xs = (xin.double() * rs.double().view(B, H, W, 1)).permute(0, 3, 1, 2)
    (F.conv_transpose2d(xs, w, stride=2) * dY.double().permute(0, 3, 1, 2)).sum().backward()
    assert torch.allclose(ref.view(2, 2, c0, N).permute(3, 2, 0, 1), w.grad, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("C,L,offset,shifts", [(64, 64, 0, [0, 8, 16, 24, 32]), (80, 24, 28, [-16, 0, 16, 40]),
                                               (48, 16, 0, [0, 16, 32, 40])])
def test_checker_match_bwd_reference_is_autograd(C, L, offset, shifts):
    """With exact forward scores, the kernel's backward formula is the gradient autograd takes through the oracle."""
    g_ = _gen(10)
    B, H, W = 2, 3, 4
    R, P = len(shifts), H * W
    x = torch.randn(B, C, H, W, generator=g_, dtype=F64)
    gd = torch.randn(B, L, generator=g_, dtype=F64)
    mask = 0b1011 if R >= 4 else (1 << R) - 1
    sel = [i for i in range(R) if (mask >> i) & 1]
    ds, dscl = torch.randn(B, R, H, W, generator=g_, dtype=F64), torch.randn(B, R, H, W, generator=g_, dtype=F64)
    dmax, dxh = torch.randn(B, 1, H, W, generator=g_, dtype=F64), torch.randn(B, C, H, W, generator=g_, dtype=F64)
    xr, gr = x.clone().requires_grad_(True), gd.clone().requires_grad_(True)
    s = orc.match_level(xr, gr, shifts, 1, offset != 0)
    loss = (s * (ds + dscl)).sum() + (s[:, sel].max(dim=1, keepdim=True)[0] * dmax).sum() + (orc.l2_normalize(xr) * dxh).sum()
    loss.backward()
    dx, Sdx, dg, Sdg = match_bwd_reference(x.permute(0, 2, 3, 1).reshape(B, P, C), gd, offset, shifts, mask,
                                           s.detach().reshape(B, R, P), ds.reshape(B, R, P),
                                           dscl.permute(0, 2, 3, 1).reshape(B, P, R), dmax.reshape(B, P),
                                           dxh.permute(0, 2, 3, 1).reshape(B, P, C))
    assert torch.allclose(dx, xr.grad.permute(0, 2, 3, 1).reshape(B, P, C), rtol=1e-10, atol=1e-12)
    assert torch.allclose(dg, gr.grad, rtol=1e-10, atol=1e-12)
    assert bool((Sdx >= dx.abs() * (1 - 1e-12)).all()) and bool((Sdg >= dg.abs() * (1 - 1e-12)).all())


def test_checker_match_reference_rounds_the_descriptor_like_the_kernel():
    """round_g: numerator with the bf16 descriptor, denominator with the fp32 norm (match_tcgen05.cu)."""
    g_ = _gen(11)
    x = _bf16(torch.randn(1, 32, 2, 3, generator=g_)).float()
    gd = torch.randn(1, 32, generator=g_)
    ref, S = match_reference(x, gd, 0, [0, 8], round_g=True)
    gb = gd.to(torch.bfloat16).double()
    num = (x.double()[0, :, 1, 2] * gb[0]).sum()
    assert torch.allclose(ref[0, 0, 1, 2], num / (x.double()[0, :, 1, 2].norm() * gd.double().norm()), rtol=1e-12)
    assert bool((S >= ref.abs() * (1 - 1e-12)).all()) and bool((S <= 1 + 1e-9).all())
