"""Training-mode execution of the post-encoder path (BASELINE.json configs[4]; reference train_VIGOR.py:120-150).

`PostEncoderFunction` is ONE `torch.autograd.Function` for everything after the two encoders: its forward is the same
sequence of C-ABI calls as inference (`PostEncoderPipeline.run`, with the intermediates kept), its backward walks that
sequence in reverse through the library's backward operators:

  * data gradients of the convolutions  = `ccvpe_igemm` on re-laid-out weights (3x3 conv <-> 3x3 conv with flipped,
    transposed weights; k2 s2 transposed conv <-> k2 s2 conv) -- on tcgen05 in the bf16 path;
  * weight gradients                    = `ccvpe_wgrad`; bias / rank-1 weight gradients = `ccvpe_colsum`;
  * ReLU mask, orientation-field normalise backward, matching + F.normalize backward, ground-head backward: own kernels.

The encoders stay PyTorch autograd (north_star), so the Function's inputs are the two encoder feature volumes, the five
aerial skip tensors (each passed TWICE -- once per decoder -- so that autograd, not this file, sums the two gradients) and
the 98 head / decoder parameters; its outputs are the reference's 9-tuple (the heatmap is marked non-differentiable: no
reference loss reads it, train_VIGOR.py:137-144).  There is no PyTorch fallback: a missing kernel raises.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import cabi
from .decoder import SCORES_CL_PAD, Fork, PostEncoderPipeline, _cl
from .specs import ENCODER_CHANNELS, SKIP_BLOCKS

GRAD_PAD = 8      # incoming 1- / 2-channel gradients (logits, orientation field) are zero padded to 8 channels


def _pad_rows(t: torch.Tensor, rows: int) -> torch.Tensor:
    """Zero-pads dim 0 of `t` to `rows`."""
    if t.shape[0] == rows:
        return t
    pad = torch.zeros((rows - t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    return torch.cat([t, pad], dim=0)


class BackwardWeights:
    """Derived, non-persistent re-layouts of the parameters for the data-gradient GEMMs (rebuilt with the forward cache)."""

    def __init__(self, pipeline: PostEncoderPipeline, dtype: torch.dtype):
        params = pipeline._params()
        spec = pipeline.spec
        tc = dtype == torch.bfloat16

        def conv_dgrad(name: str) -> dict:
            """3x3 pad-1 conv [Cout, Cin, 3, 3] -> the 3x3 pad-1 conv that maps dY [.., pad8(Cout)] to dX [.., Cin]."""
            W = params[name + ".weight"].detach()
            cout, cin = W.shape[0], W.shape[1]
            Wf = _pad_rows(W.flip(2, 3), -(-cout // GRAD_PAD) * GRAD_PAD)          # [Cout_p, Cin, 3, 3]
            coutp = Wf.shape[0]
            out = dict(w_kn=Wf.permute(2, 3, 0, 1).reshape(9, coutp, cin).to(dtype).contiguous(), bias=None, cout=cin,
                       k=coutp)
            if tc:
                out["w_nk"] = cabi.w_nk_layout(Wf.permute(1, 2, 3, 0).reshape(cin, 9, coutp), [coutp])
            return out

        def deconv_dgrad(name: str, lead: int, lead_pad: int) -> dict:
            """ConvTranspose2d(k2, s2) [Cin, Cout, 2, 2] -> the k2 s2 conv that maps dY [.., Cout] to dX.  Column order of
            dX: lead == -1 (localisation decoder): [the C map channels | 8 columns whose first is d(max score)];
            lead > 0 (orientation decoder, level 1): [lead_pad score columns | the C map channels]."""
            W = params[name + ".weight"].detach()                                    # [Cin, Cout, 2, 2]
            cout = W.shape[1]
            if lead == -1:
                extra = torch.zeros((GRAD_PAD,) + tuple(W.shape[1:]), dtype=W.dtype, device=W.device)
                extra[0] = W[0]
                W = torch.cat([W[1:], extra], dim=0)
            elif lead > 0:
                pad = torch.zeros((lead_pad - lead,) + tuple(W.shape[1:]), dtype=W.dtype, device=W.device)
                W = torch.cat([W[:lead], pad, W[lead:]], dim=0)
            n = W.shape[0]
            out = dict(w_kn=W.permute(2, 3, 1, 0).reshape(4, cout, n).to(dtype).contiguous(), bias=None, cout=n, k=cout)
            if tc:
                out["w_nk"] = cabi.w_nk_layout(W.permute(0, 2, 3, 1).reshape(n, 4, cout), [cout])
            return out

        self.loc: List[dict] = []
        self.ori: List[dict] = []
        for i, n in enumerate(range(6, 0, -1)):
            for branch, sfx in ((self.loc, ""), (self.ori, "_ori")):
                lead = -1 if sfx == "" else (spec.n_rolls if n == 6 else 0)
                branch.append(dict(deconv=deconv_dgrad("deconv%d%s" % (n, sfx), lead, SCORES_CL_PAD),
                                   conv_a=conv_dgrad("conv%d%s.0" % (n, sfx)),
                                   conv_b=conv_dgrad("conv%d%s.2" % (n, sfx))))
        # aerial cell descriptors: conv k2 s2 (Linear over 2x2 cells) -> its data gradient is a k2 s2 transposed conv
        lw = params["sat_feature_to_descriptors.1.weight"].detach()
        D = lw.shape[0]
        Wc = lw.view(D, ENCODER_CHANNELS, 2, 2)
        self.cell = dict(w_kn=Wc.permute(0, 2, 3, 1).reshape(1, D, 4 * ENCODER_CHANNELS).to(dtype).contiguous(), bias=None,
                         cout=ENCODER_CHANNELS)
        if tc:
            self.cell["w_nk"] = cabi.w_nk_layout(Wc.permute(2, 3, 1, 0).reshape(4 * ENCODER_CHANNELS, 1, D), [D])


class PostEncoderTrainer:
    """Forward-with-save and backward of one `PostEncoderPipeline`."""

    def __init__(self, pipeline: PostEncoderPipeline):
        self.p = pipeline
        self._bwd: Dict[torch.dtype, BackwardWeights] = {}
        self._bwd_sig = None

    def _bwd_weights(self, dtype: torch.dtype) -> BackwardWeights:
        self.p._weights(dtype)                       # refreshes pipeline._sig
        if self._bwd_sig != self.p._sig:
            self._bwd.clear()
            self._bwd_sig = self.p._sig
        if dtype not in self._bwd:
            self._bwd[dtype] = BackwardWeights(self.p, dtype)
        return self._bwd[dtype]

    # -- operator helpers ---------------------------------------------------------------------------------------
    def _wgrad(self, tag, a0, c0, a1, c1, geom, g2d, N, row_scale, dtype) -> torch.Tensor:
        """geom = (B, Hin, Win, Hout, Wout, stride, k, pad).  Returns fp32 [taps, c0 + c1, N]."""
        B, Hin, Win, Hout, Wout, stride, k, pad = geom
        d = cabi.WgradDesc()
        d.a0, d.a1 = a0.data_ptr(), (a1.data_ptr() if a1 is not None else None)
        d.c0, d.c1 = c0, c1
        d.ld0, d.ld1 = a0.stride(-2), (a1.stride(-2) if a1 is not None else 0)
        d.B, d.Hin, d.Win, d.Hout, d.Wout = B, Hin, Win, Hout, Wout
        d.stride, d.kh, d.kw, d.pad = stride, k, k, pad
        d.g, d.N, d.ldg = g2d.data_ptr(), N, g2d.stride(-2)
        d.g_row_scale = row_scale.data_ptr() if row_scale is not None else None
        d.dtype = cabi.dtype_code(dtype)
        out = torch.empty((k * k, c0 + c1, N), dtype=torch.float32, device=a0.device)
        d.out = out.data_ptr()
        d.backend = self.p.backend
        n_ws = cabi.wgrad_workspace_elems(d)
        ws = torch.empty(n_ws, dtype=torch.float32, device=a0.device)
        d.workspace, d.workspace_elems = ws.data_ptr(), n_ws
        M = B * Hout * Wout
        if self.p.timer is not None:
            tag = cabi.wgrad_kernel_name(d) + ":" + tag
        esz = a0.element_size()
        self.p._op(tag, 2.0 * M * N * k * k * (c0 + c1),
                   (B * Hin * Win * (c0 + c1) + M * N) * esz + k * k * (c0 + c1) * N * 4, lambda: cabi.wgrad(d))
        return out

    def _colsum(self, x, C_, w=None, s=1) -> torch.Tensor:
        out = torch.empty((s * s, C_), dtype=torch.float32, device=x.device)
        view = x if x.stride(-2) == x.shape[-1] else None
        if view is None:                                   # channel slice of a wider tensor: hand the kernel the real stride
            B, H, W, _ = x.shape
            view = x.as_strided((B, H, W, x.stride(-2)), (x.stride(0), x.stride(1), x.stride(2), 1))
        self.p._op("colsum_partial_kernel:colsum|", 2.0 * view.numel(), view.numel() * view.element_size(),
                   lambda: cabi.colsum(view, C_, out, w, s))
        return out

    def _conv_bwd(self, name, wt_bwd, a0, a1, dY, n_real, dtype, grads, pname):
        """3x3 conv backward: weight / bias gradients into `grads`, returns dX [B, H, W, c0 + c1] (dtype)."""
        B, H, W, c0 = a0.shape
        c1 = a1.shape[-1] if a1 is not None else 0
        kp = wt_bwd["k"]                                   # channels of dY (padded to 8)
        geom = (B, H, W, H, W, 1, 3, 1)
        dw = self._wgrad("wgrad|" + name, a0, c0, a1, c1, geom, dY.view(B * H * W, kp), kp, None, dtype)
        grads[pname + ".weight"] = dw.view(3, 3, c0 + c1, kp)[..., :n_real].permute(3, 2, 0, 1)
        grads[pname + ".bias"] = self._colsum(dY, kp)[0, :n_real]
        dX = torch.empty((B, H, W, c0 + c1), dtype=dtype, device=a0.device)
        self.p._igemm("igemm:dgrad_conv3x3|" + name, dY, kp, None, 0, B, H, W, H, W, 1, 3, 1, c0 + c1, dtype, wt_bwd, dX, 0,
                      c0 + c1)
        return dX

    def _deconv_bwd(self, name, wt_bwd, srcs, d_up, cout, dtype, grads, pname, row_scale=None, mx=None):
        """k2 s2 transposed conv backward.  srcs: [(tensor [B, H, W, ld], n_real_channels, first weight row)], d_up: a view
        [B, 2H, 2W, cout] (row stride may exceed cout).  Returns dIn [B, H, W, N'] in wt_bwd's column order."""
        B, H2, W2, _ = d_up.shape
        H, W = H2 // 2, W2 // 2
        geom = (B, H2, W2, H, W, 2, 2, 0)
        pw = torch.empty_like(self.p._params()[pname + ".weight"], dtype=torch.float32)      # [Cin, Cout, 2, 2]
        if row_scale is not None and dtype == torch.bfloat16 and self.p.backend != cabi.BACKEND_SIMT:
            # tensor-core weight gradient: its G operand is the normalised map itself (one small HBM-bound pass)
            scaled = []
            for src, n_real, row0 in srcs:
                xh = torch.empty_like(src)
                self.p._op("scale_rows_kernel:scale_rows|" + name, src.numel(), 2.0 * src.numel() * src.element_size(),
                           lambda s_=src, o_=xh: cabi.scale_rows(s_, row_scale, o_))
                scaled.append((xh, n_real, row0))
            srcs, row_scale = scaled, None
        for src, n_real, row0 in srcs:
            ld = src.shape[-1]
            dw = self._wgrad("wgrad|" + name, d_up, cout, None, 0, geom, src.view(B * H * W, ld), ld, row_scale, dtype)
            pw[row0:row0 + n_real] = dw.view(2, 2, cout, ld)[..., :n_real].permute(3, 2, 0, 1)
        if mx is not None:                                   # the max-score channel (row 0 of the weight)
            pw[0] = self._colsum(d_up, cout, w=mx, s=2).view(2, 2, cout).permute(2, 0, 1)
        grads[pname + ".weight"] = pw
        grads[pname + ".bias"] = self._colsum(d_up, cout)[0]
        n_out = wt_bwd["cout"]
        d_in = torch.empty((B, H, W, n_out), dtype=dtype, device=d_up.device)
        d = dict(wt_bwd)
        self._igemm_strided("igemm:dgrad_deconv|" + name, d_up, cout, B, H2, W2, H, W, 2, 2, 0, n_out, dtype, d, d_in)
        return d_in

    def _igemm_strided(self, tag, a0, c0, B, Hin, Win, Hout, Wout, stride, k, pad, N, dtype, wt, out, out_mode=0, ldo=None):
        """`PostEncoderPipeline._igemm` for a source that is a channel slice of a wider tensor (row stride != c0)."""
        p = self.p
        d = cabi.IgemmDesc()
        d.a0, d.a1 = a0.data_ptr(), None
        d.c0, d.c1, d.ld0, d.ld1 = c0, 0, a0.stride(-2), 0
        d.B, d.Hin, d.Win, d.Hout, d.Wout = B, Hin, Win, Hout, Wout
        d.stride, d.kh, d.kw, d.pad = stride, k, k, pad
        d.N, d.dtype = N, cabi.dtype_code(dtype)
        d.w_kn = wt["w_kn"].data_ptr()
        d.w_nk = wt["w_nk"].data_ptr() if "w_nk" in wt else None
        d.bias = d.row_scale = d.row_r1 = d.r1_w = None
        d.relu, d.out_mode, d.out_dtype = 0, out_mode, cabi.dtype_code(out.dtype)
        d.ldo = N if ldo is None else ldo
        d.out = out.data_ptr()
        d.backend = p.backend
        M, K = B * Hout * Wout, k * k * c0
        if p.timer is not None:
            tag = cabi.igemm_kernel_name(d) + ":" + tag
        esz = a0.element_size()
        p._op(tag, 2.0 * M * N * K, (B * Hin * Win * c0 + K * N) * esz + M * N * out.element_size(), lambda: cabi.igemm(d))

    # -- forward ------------------------------------------------------------------------------------------------
    def forward(self, grd_feat, sat_feat, multiscale, dtype) -> Tuple[Tuple[torch.Tensor, ...], dict]:
        saved: dict = {}
        out = self.p.run(grd_feat, sat_feat, multiscale, dtype, save=saved)
        return out, saved

    # -- backward -----------------------------------------------------------------------------------------------
    @torch.no_grad()
    def backward(self, sv: dict, d_logits: Optional[torch.Tensor], d_ori: Optional[torch.Tensor],
                 d_scores: Sequence[Optional[torch.Tensor]]):
        """Returns (d_grd_feat fp32 NCHW, d_sat_feat channels-last, [d_skip loc x5], [d_skip ori x5], {param name: grad})."""
        p = self.p
        spec = p.spec
        dtype = sv["dtype"]
        B = sv["B"]
        dev = sv["fs"].device
        w = p._weights(dtype)
        wb = self._bwd_weights(dtype)
        grads: Dict[str, torch.Tensor] = {}
        skips = sv["skips"]
        Hh, Wh = sv["o_raw"].shape[1:3]
        D = spec.sat_dim

        # ---- orientation decoder (reference models.py:322-341), output -> bottleneck ----
        # (on a forked side stream: independent of the localisation decoder's backward until the bottleneck level)
        fork = Fork(dev, enabled=p.timer is None and p.concurrent)
        with fork:
            d_sk_ori: List[Optional[torch.Tensor]] = [None] * 5
            dY = torch.empty((B, Hh, Wh, GRAD_PAD), dtype=dtype, device=dev)
            if d_ori is None:
                dY.zero_()
            else:
                do = d_ori.contiguous().float()
                p._op("ori_normalize_bwd_kernel:ori_normalize_bwd|", 12.0 * B * Hh * Wh, B * Hh * Wh * (16 + 8 * dY.element_size()),
                      lambda: cabi.ori_normalize_bwd(sv["o_raw"], do, dY))
            d_ori_in = None
            for l in range(5, -1, -1):
                rec, wl = sv["ori"][l], wb.ori[l]
                n = 6 - l
                nm = "ori%d" % n
                h, up = rec["h"], rec["up"]
                n_real = 2 if l == 5 else spec.ori_conv_out[l]
                dh = self._conv_bwd(nm + "b", wl["conv_b"], h, None, dY, n_real, dtype, grads, "conv%d_ori.2" % n)
                p._op("relu_bwd_kernel:relu_bwd|" + nm, dh.numel(), 3.0 * dh.numel() * dh.element_size(),
                      lambda: cabi.relu_bwd(dh, h))
                skip = skips[l] if l < 5 else None
                dcat = self._conv_bwd(nm + "a", wl["conv_a"], up, skip, dh, h.shape[-1], dtype, grads, "conv%d_ori.0" % n)
                cout = up.shape[-1]
                if skip is not None:
                    d_sk_ori[l] = dcat[..., cout:]
                d_up = dcat[..., :cout]
                if l == 0:
                    srcs = [(sv["scores_cl"], spec.n_rolls, 0), (sv["xhat"], D, spec.n_rolls)]
                else:
                    srcs = [(rec["inp"], rec["inp"].shape[-1], 0)]
                d_in = self._deconv_bwd(nm, wl["deconv"], srcs, d_up, cout, dtype, grads, "deconv%d_ori" % n)
                if l == 0:
                    d_ori_in = d_in                               # [B, 8, 8, 32 + D]: d scores_1 | d xhat_1
                else:
                    dY = d_in

        # ---- localisation decoder (reference models.py:186-320), output -> bottleneck ----
        d_sk_loc: List[Optional[torch.Tensor]] = [None] * 5
        dgs: List[torch.Tensor] = [None] * 6
        dY = torch.empty((B, Hh, Wh, GRAD_PAD), dtype=dtype, device=dev)
        if d_logits is None:
            dY.zero_()
        else:
            dl = d_logits.contiguous().float().view(B, 1, Hh * Wh)
            p._op("planar_to_cl_kernel:planar_to_cl|", 0.0, B * Hh * Wh * (4 + 8 * dY.element_size()),
                  lambda: cabi.planar_to_cl(dl, dY))
        for l in range(5, -1, -1):
            rec, wl = sv["loc"][l], wb.loc[l]
            n = 6 - l
            nm = "loc%d" % n
            h, up, x = rec["h"], rec["up"], rec["x"]
            n_real = 1 if l == 5 else spec.loc_conv_out[l]
            dh = self._conv_bwd(nm + "b", wl["conv_b"], h, None, dY, n_real, dtype, grads, "conv%d.2" % n)
            p._op("relu_bwd_kernel:relu_bwd|" + nm, dh.numel(), 3.0 * dh.numel() * dh.element_size(),
                  lambda: cabi.relu_bwd(dh, h))
            skip = skips[l] if l < 5 else None
            dcat = self._conv_bwd(nm + "a", wl["conv_a"], up, skip, dh, h.shape[-1], dtype, grads, "conv%d.0" % n)
            cout = up.shape[-1]
            if skip is not None:
                d_sk_loc[l] = dcat[..., cout:]
            d_up = dcat[..., :cout]
            C = x.shape[-1]
            d_in = self._deconv_bwd(nm, wl["deconv"], [(x, C, 1)], d_up, cout, dtype, grads, "deconv%d" % n,
                                    row_scale=rec["inv"], mx=rec["mx"])            # [B, H, W, C + 8]
            # matching + F.normalize backward (a4-a6): d scores (loss + orientation decoder) + d max + d xhat -> d x, d g
            _, H, W, _ = x.shape
            dx = torch.empty_like(x)
            g_l = sv["g"][l]
            dg = torch.empty_like(g_l)
            ds = d_scores[l]
            ds = ds.contiguous().float() if ds is not None else None
            d2 = d_in.view(B * H * W, C + GRAD_PAD)
            ds_cl = dxh2 = None
            if l == 0:      # the orientation decoder's gradients are needed from here on
                fork.join(d_ori_in, *[t for t in d_sk_ori if t is not None], *[grads[k] for k in grads if "_ori" in k])
            if l == 0 and d_ori_in is not None:
                o2 = d_ori_in.view(B * H * W, SCORES_CL_PAD + D)
                ds_cl, dxh2 = o2, o2[:, SCORES_CL_PAD:]
            R = len(rec["shifts"])
            p._op("match_level_bwd_kernel:match_bwd|l%d" % (l + 1), 4.0 * R * g_l.shape[1] * B * H * W,
                  3.0 * x.numel() * x.element_size() + 2.0 * R * B * H * W * 4,
                  lambda: cabi.match_level_bwd(x, g_l, rec["offset"], rec["shifts"], rec["mask"], rec["scores"], ds, ds_cl,
                                               d2[:, C:], d2, dxh2, dx, dg))
            dgs[l] = dg
            dY = dx

        # ---- aerial cell descriptors (models.py:102-104, 173-184) ----
        fs = sv["fs"]
        Hs, Ws = fs.shape[1], fs.shape[2]
        d_x1 = dY                                                                      # [B, 8, 8, D]
        geom = (B, Hs, Ws, Hs // 2, Ws // 2, 2, 2, 0)
        dw = self._wgrad("wgrad|cell", fs, ENCODER_CHANNELS, None, 0, geom, d_x1.view(B * (Hs // 2) * (Ws // 2), D), D, None,
                         dtype)
        grads["sat_feature_to_descriptors.1.weight"] = dw.view(2, 2, ENCODER_CHANNELS, D).permute(3, 2, 0, 1).reshape(D, -1)
        grads["sat_feature_to_descriptors.1.bias"] = self._colsum(d_x1, D)[0]
        d_fs = torch.empty((B, Hs, Ws, ENCODER_CHANNELS), dtype=dtype, device=dev)
        self._igemm_strided("igemm:dgrad_cell|", d_x1, D, B, Hs // 2, Ws // 2, Hs // 2, Ws // 2, 1, 1, 0, 4 * ENCODER_CHANNELS,
                            dtype, wb.cell, d_fs, out_mode=1, ldo=ENCODER_CHANNELS)

        # ---- ground descriptor heads (models.py:57-97, 152-157) ----
        grd_feat = sv["grd_feat"]
        heads = w["heads"]
        d_fg = torch.empty(tuple(grd_feat.shape), dtype=torch.float32, device=dev)
        dw1 = [torch.empty_like(hd[0]) for hd in heads]
        db1 = [torch.empty_like(hd[1]) for hd in heads]
        dw2 = [torch.empty_like(hd[2]) for hd in heads]
        db2 = [torch.empty_like(hd[3]) for hd in heads]
        p._op("heads_bwd_data_kernel:grd_descriptors_bwd|", 4.0 * grd_feat.numel() * 126,
              2.0 * grd_feat.numel() * 4, lambda: cabi.grd_descriptors_bwd(grd_feat, heads, dgs, d_fg, dw1, db1, dw2, db2))
        params = p._params()
        for l in range(6):
            base = "grd_feature_to_descriptor%d" % (l + 1)
            grads[base + ".0.weight"] = dw1[l].view_as(params[base + ".0.weight"])
            grads[base + ".0.bias"] = db1[l]
            grads[base + ".2.weight"] = dw2[l].view_as(params[base + ".2.weight"])
            grads[base + ".2.bias"] = db2[l].view_as(params[base + ".2.bias"])
        return d_fg, d_fs, d_sk_loc, d_sk_ori, grads


class PostEncoderFunction(torch.autograd.Function):
    """inputs: trainer, dtype, grd_feat, sat_feat, 5 skips (localisation decoder), the same 5 skips (orientation decoder),
    then the decoder parameters in `trainer.p._params()` order."""

    @staticmethod
    def forward(ctx, trainer: PostEncoderTrainer, dtype, grd_feat, sat_feat, *rest):
        skips = rest[:5]
        multiscale = [None] * (max(SKIP_BLOCKS) + 1)
        for i, blk in enumerate(SKIP_BLOCKS):
            multiscale[blk] = skips[i]
        with cabi.device_of(sat_feat):
            out, saved = trainer.forward(grd_feat.detach(), sat_feat.detach(), multiscale, dtype)
        ctx.trainer, ctx.saved = trainer, saved
        ctx.param_names = list(trainer.p._params().keys())
        ctx.in_dtypes = (grd_feat.dtype, sat_feat.dtype, [s.dtype for s in skips])
        ctx.mark_non_differentiable(out[1])
        return tuple(out)

    @staticmethod
    def backward(ctx, *gouts):
        trainer, sv = ctx.trainer, ctx.saved
        d_logits, _d_heat, d_ori = gouts[0], gouts[1], gouts[2]
        with cabi.device_of(sv["fs"]):
            d_fg, d_fs, d_sk_loc, d_sk_ori, grads = trainer.backward(sv, d_logits, d_ori, gouts[3:9])
        ctx.saved = None
        gdt, sdt, kdt = ctx.in_dtypes
        res = [None, None, d_fg.to(gdt), d_fs.permute(0, 3, 1, 2).to(sdt)]
        res += [t.permute(0, 3, 1, 2).to(dt) for t, dt in zip(d_sk_loc, kdt)]
        res += [t.permute(0, 3, 1, 2).to(dt) for t, dt in zip(d_sk_ori, kdt)]
        res += [grads[k] for k in ctx.param_names]
        return tuple(res)


class GraphedTrainStep:
    """One whole training step -- zero_grad, forward, losses, backward, gradient all-reduce, optimizer step -- captured in a
    single CUDA graph and replayed (the eager step is bound by ~3000 host-side launches of small encoder / optimizer /
    decoder kernels, not by the GPU).  Everything in the step is capturable: the library never allocates or synchronises, its
    tensor maps are by-value kernel parameters, the derived weight caches are rebuilt by kernels that are part of the
    captured graph, the gradient buckets are static memory, and the optimizer must be constructed with capturable=True.

        step = GraphedTrainStep(lambda grd, sat, gt, gwo, gor: ..., example_inputs)    # closure returns the loss tensor
        loss = step(grd, sat, gt, gwo, gor)                                             # copies inputs in, replays

    `fn` is run `warmup` times eagerly on a side stream before capture (so every lazily-built cache, cuDNN plan and
    optimizer state exists): `warmup` real optimizer steps happen during construction; the capture itself executes nothing."""

    def __init__(self, fn, example_inputs: Sequence[torch.Tensor], warmup: int = 3):
        self.static_in = [t.clone() for t in example_inputs]
        dev = self.static_in[0].device
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(warmup):
                fn(*self.static_in)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        n0 = cabi.launch_count()
        with torch.cuda.graph(self.graph):
            self.static_loss = fn(*self.static_in)
        self.launches = cabi.launch_count() - n0          # libccvpe_b200 kernels inside one replay
        cabi.add_replayed_launches(-self.launches)        # captured, not executed

    def __call__(self, *inputs: torch.Tensor) -> torch.Tensor:
        for dst, src in zip(self.static_in, inputs):
            if dst.data_ptr() != src.data_ptr():
                dst.copy_(src, non_blocking=True)
        self.graph.replay()
        cabi.add_replayed_launches(self.launches)
        return self.static_loss
