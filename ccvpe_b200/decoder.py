"""Host-side orchestration of the CUDA hot path: everything `CVM_*.forward` does after the two encoders.

One `PostEncoderPipeline` per model instance.  It owns (a) a derived, non-persistent cache of re-laid-out weights
(the module's parameters keep the reference's shapes and names so checkpoints load strictly; the cache is rebuilt
whenever a parameter's version counter or storage changes) and (b) the sequence of C-ABI calls.  There is no
PyTorch or CPU fallback in here: every stage is a kernel of libccvpe_b200.so.

Data layout in HBM: activations are channels-last [B, H, W, C] in the pipeline dtype (fp32 parity path, bf16
throughput path); nothing is ever concatenated -- `cat([max, normalize(x)])` becomes a row-scale + rank-1 epilogue of
the transposed-conv GEMM and `cat([x, skip])` a K-split over two sources of the conv GEMM.  The nine tensors handed
back to the caller are fp32 in the reference's NCHW shapes (reference models.py:343).
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import cabi
from .specs import ENCODER_CHANNELS, SKIP_BLOCKS, SKIP_CHANNELS, VariantSpec, loc_roll_indices

SCORES_CL_PAD = 32  # channel stride of the channels-last copy of the level-1 score volume (ori decoder input)


def _cl(t: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """Logical NCHW tensor -> channels-last [B, H, W, C] contiguous in `dtype` (free if it already is)."""
    v = t.permute(0, 2, 3, 1)
    if v.dtype != dtype:
        v = v.to(dtype)
    return v.contiguous()


_SIDE_STREAMS: Dict[int, "torch.cuda.Stream"] = {}


class Fork:
    """Runs a block of launches on a side stream that forks from / joins into the current stream, so that two independent
    kernel sequences (localisation vs orientation decoder, ground vs aerial encoder) execute concurrently.  Matters at small
    batches, where single kernels do not fill the 148 SMs; inside a CUDA-graph capture the fork / join become graph edges.

        fork = Fork(device, enabled)
        with fork:            # launches in here go to the side stream
            ...
        ...                   # launches on the main stream, concurrent with the block above
        fork.join(t1, t2)     # main waits for the side stream; tensors produced there are handed over to main

    Tensors allocated in the block belong to the side stream's pool: pass the ones that outlive the call to `join`
    (outside graph capture they are `record_stream`-ed on the main stream; main-stream tensors read in the block are kept
    alive by the caller until `join`)."""

    def __init__(self, device, enabled: bool = True):
        self.enabled = bool(enabled)
        self.device = device
        if self.enabled:
            idx = device.index if device.index is not None else torch.cuda.current_device()
            if idx not in _SIDE_STREAMS:
                _SIDE_STREAMS[idx] = torch.cuda.Stream(device=device)
            self.side = _SIDE_STREAMS[idx]
            self.main = torch.cuda.current_stream(device)
            self._ctx = None

    def __enter__(self):
        if self.enabled:
            self.side.wait_stream(self.main)
            self._ctx = torch.cuda.stream(self.side)
            self._ctx.__enter__()
        return self

    def __exit__(self, *exc):
        if self.enabled:
            self._ctx.__exit__(*exc)
        return False

    def join(self, *tensors):
        if not self.enabled:
            return
        self.main.wait_stream(self.side)
        if not torch.cuda.is_current_stream_capturing():
            for t in tensors:
                if t is not None:
                    t.record_stream(self.main)


class OpTimer:
    """Optional per-operator CUDA-event timer (bench.py): events are recorded on torch's current stream, which is the
    stream every kernel of the pipeline is launched on.  `flops` / `nbytes` are the ALGORITHMIC work of the call."""

    def __init__(self):
        self.records = []

    def run(self, tag: str, flops: float, nbytes: float, fn):
        s = torch.cuda.Event(enable_timing=True)
        e = torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        self.records.append((tag, s, e, float(flops), float(nbytes)))

    def summary(self) -> Dict[str, dict]:
        torch.cuda.synchronize()
        out: Dict[str, dict] = {}
        for tag, s, e, fl, nb in self.records:
            r = out.setdefault(tag, dict(launches=0, ms=0.0, flops=0.0, bytes=0.0))
            r["launches"] += 1
            r["ms"] += s.elapsed_time(e)
            r["flops"] += fl
            r["bytes"] += nb
        return out


class PostEncoderPipeline:
    def __init__(self, module: torch.nn.Module, spec: VariantSpec, ori_noise: Optional[float] = None):
        self._module = [module]          # list: do not register the owner as a sub-module
        self.spec = spec
        self.ori_noise = ori_noise
        self.backend = cabi.BACKEND_AUTO
        self.concurrent = True           # run independent branches (orientation / localisation decoder) on forked streams
        self._cache: Dict[torch.dtype, dict] = {}
        self._sig = None
        self.timer: Optional[OpTimer] = None

    def _op(self, tag: str, flops: float, nbytes: float, fn):
        if self.timer is None:
            fn()
        else:
            self.timer.run(tag, flops, nbytes, fn)

    # -- derived weight cache ---------------------------------------------------------------------------------
    def _params(self) -> Dict[str, torch.Tensor]:
        return {k: v for k, v in self._module[0].named_parameters()
                if not k.startswith(("grd_efficientnet.", "sat_efficientnet."))}

    def _signature(self, params):
        return tuple((k, p.data_ptr(), p._version, p.device) for k, p in params.items())

    @torch.no_grad()
    def _weights(self, dtype: torch.dtype) -> dict:
        params = self._params()
        sig = self._signature(params)
        if sig != self._sig:
            self._cache.clear()
            self._sig = sig
        if dtype in self._cache:
            return self._cache[dtype]
        spec = self.spec
        f32 = lambda t: t.detach().to(torch.float32).contiguous()
        w: dict = {}
        # a1 ground heads
        w["heads"] = []
        for l in range(1, 7):
            w1 = params["grd_feature_to_descriptor%d.0.weight" % l]
            w["heads"].append((f32(w1.reshape(w1.shape[0], -1)),
                               f32(params["grd_feature_to_descriptor%d.0.bias" % l]),
                               f32(params["grd_feature_to_descriptor%d.2.weight" % l].reshape(-1)),
                               f32(params["grd_feature_to_descriptor%d.2.bias" % l])))
        # a3 aerial cell descriptors: Linear(5120 -> D) with the 5120 axis ordered (c, dh, dw) == conv k2 s2
        lw = params["sat_feature_to_descriptors.1.weight"].detach()
        D = lw.shape[0]
        tc = dtype == torch.bfloat16     # also build the K-major layout of the tcgen05 backend
        w["cell"] = dict(w_kn=lw.view(D, ENCODER_CHANNELS, 2, 2).permute(2, 3, 1, 0).reshape(4, ENCODER_CHANNELS, D)
                         .to(dtype).contiguous(), bias=f32(params["sat_feature_to_descriptors.1.bias"]))
        if tc:
            w["cell"]["w_nk"] = cabi.w_nk_layout(
                lw.view(D, ENCODER_CHANNELS, 2, 2).permute(0, 2, 3, 1).reshape(D, 4, ENCODER_CHANNELS), [ENCODER_CHANNELS])

        def deconv(name: str, lead: int, lead_pad: int):
            """ConvTranspose2d weight [Cin, Cout, 2, 2] -> GEMM B [1][K][4*Cout], N ordered (i, j, co).
            lead > 0: the first `lead` input channels are a separate source padded to `lead_pad` channels;
            lead == -1: the first input channel (the max score) becomes the rank-1 epilogue vector."""
            W = params[name + ".weight"].detach()
            cout = W.shape[1]
            out = dict(bias=f32(params[name + ".bias"].detach().repeat(4)), cout=cout)
            if lead == -1:
                out["r1_w"] = f32(W[0].permute(1, 2, 0).reshape(4 * cout))
                W = W[1:]
            elif lead > 0:
                pad = torch.zeros((lead_pad - lead,) + tuple(W.shape[1:]), dtype=W.dtype, device=W.device)
                W = torch.cat([W[:lead], pad, W[lead:]], dim=0)
            out["w_kn"] = W.permute(0, 2, 3, 1).reshape(1, W.shape[0], 4 * cout).to(dtype).contiguous()
            if tc:
                rows = W.permute(2, 3, 1, 0).reshape(4 * cout, 1, W.shape[0])
                out["w_nk"] = cabi.w_nk_layout(rows, [lead_pad, W.shape[0] - lead_pad] if lead > 0 else [W.shape[0]])
            return out

        def conv(name: str, c0: int):
            W = params[name + ".weight"].detach()        # [Cout, Cin, 3, 3]
            out = dict(w_kn=W.permute(2, 3, 1, 0).reshape(9, W.shape[1], W.shape[0]).to(dtype).contiguous(),
                       bias=f32(params[name + ".bias"]), cout=W.shape[0])
            if tc:
                rows = W.permute(0, 2, 3, 1).reshape(W.shape[0], 9, W.shape[1])
                out["w_nk"] = cabi.w_nk_layout(rows, [c0, W.shape[1] - c0] if c0 < W.shape[1] else [c0])
            return out

        w["loc"], w["ori"] = [], []
        for i, n in enumerate(range(6, 0, -1)):
            for branch, sfx, douts in (("loc", "", spec.loc_deconv_out), ("ori", "_ori", spec.ori_deconv_out)):
                dname = "deconv%d%s" % (n, sfx)
                if branch == "loc":
                    dc = deconv(dname, -1, 0)
                else:
                    dc = deconv(dname, spec.n_rolls if n == 6 else 0, SCORES_CL_PAD)
                ca = conv("conv%d%s.0" % (n, sfx), douts[i])          # sources: (deconv output, encoder skip)
                cb = conv("conv%d%s.2" % (n, sfx), params["conv%d%s.2.weight" % (n, sfx)].shape[1])
                w[branch].append(dict(deconv=dc, conv_a=ca, conv_b=cb))
        self._cache[dtype] = w
        return w

    # -- kernel helpers ---------------------------------------------------------------------------------------
    def _igemm(self, tag, a0, c0, a1, c1, B, Hin, Win, Hout, Wout, stride, k, pad, N, dtype, wt, out, out_mode, ldo,
               relu=False, row_scale=None, row_r1=None, r1_w=None):
        d = cabi.IgemmDesc()
        d.a0, d.a1 = a0.data_ptr(), (a1.data_ptr() if a1 is not None else None)
        d.c0, d.c1 = c0, c1
        d.ld0, d.ld1 = a0.shape[-1], (a1.shape[-1] if a1 is not None else 0)
        d.B, d.Hin, d.Win, d.Hout, d.Wout = B, Hin, Win, Hout, Wout
        d.stride, d.kh, d.kw, d.pad = stride, k, k, pad
        d.N, d.dtype = N, cabi.dtype_code(dtype)
        d.w_kn = wt["w_kn"].data_ptr()
        d.w_nk = wt["w_nk"].data_ptr() if "w_nk" in wt else None
        d.bias = wt["bias"].data_ptr() if wt.get("bias") is not None else None
        d.row_scale = row_scale.data_ptr() if row_scale is not None else None
        d.row_r1 = row_r1.data_ptr() if row_r1 is not None else None
        d.r1_w = r1_w.data_ptr() if r1_w is not None else None
        d.relu, d.out_mode, d.out_dtype, d.ldo = int(relu), out_mode, cabi.dtype_code(out.dtype), ldo
        d.out = out.data_ptr()
        d.backend = self.backend
        M, K = B * Hout * Wout, k * k * (c0 + c1)
        esz = a0.element_size()
        nbytes = (B * Hin * Win * (c0 + c1) + K * N) * esz + M * N * out.element_size()
        if self.timer is not None:            # attribute the launch to the kernel the library will pick
            tag = cabi.igemm_kernel_name(d) + ":" + tag
        self._op(tag, 2.0 * M * N * K, nbytes, lambda: cabi.igemm(d))

    def _deconv(self, wt, a0, c0, a1, c1, dtype, row_scale=None, row_r1=None, name=""):
        """ConvTranspose2d(k2, s2) as GEMM + pixel shuffle (reference models.py:109-124)."""
        B, H, W, _ = a0.shape
        cout = wt["cout"]
        out = torch.empty((B, 2 * H, 2 * W, cout), dtype=dtype, device=a0.device)
        self._igemm("igemm:deconv|" + name, a0, c0, a1, c1, B, H, W, H, W, 1, 1, 0, 4 * cout, dtype, wt, out, 1, cout,
                    row_scale=row_scale, row_r1=row_r1, r1_w=wt.get("r1_w") if row_r1 is not None else None)
        return out

    def _conv3(self, wt, a0, a1, dtype, relu, planar_f32=False, out_f32=False, name=""):
        """3x3 pad-1 conv over the K-concatenation of a0 and a1 (reference models.py:42-47)."""
        B, H, W, c0 = a0.shape
        c1 = a1.shape[-1] if a1 is not None else 0
        cout = wt["cout"]
        if planar_f32:
            out = torch.empty((B, cout, H, W), dtype=torch.float32, device=a0.device)
            mode, ldo = 2, 0
        else:
            out = torch.empty((B, H, W, cout), dtype=torch.float32 if out_f32 else dtype, device=a0.device)
            mode, ldo = 0, cout
        self._igemm("igemm:conv3x3|" + name, a0, c0, a1, c1, B, H, W, H, W, 1, 3, 1, cout, dtype, wt, out, mode, ldo, relu=relu)
        return out

    # -- the path ---------------------------------------------------------------------------------------------
    @torch.no_grad()
    def run(self, grd_feat: torch.Tensor, sat_feat: torch.Tensor, multiscale: Sequence[torch.Tensor],
            dtype: torch.dtype, save: Optional[dict] = None) -> Tuple[torch.Tensor, ...]:
        """`save`: a dict that receives every intermediate the backward pass needs (training.py)."""
        if not (grd_feat.is_cuda and sat_feat.is_cuda):
            raise cabi.CcvpeError("the post-encoder path runs on CUDA only (sm_100a); there is no CPU fallback")
        spec = self.spec
        w = self._weights(dtype)
        dev = sat_feat.device
        B = sat_feat.shape[0]
        f32 = torch.float32

        # a1 -- six ground descriptors (fp32, tiny)
        if grd_feat.dtype not in (torch.float32, torch.bfloat16):
            grd_feat = grd_feat.float()
        Bg, Kg, Hg, Wg = grd_feat.shape
        if Hg != spec.grd_feat_h:
            raise cabi.CcvpeError("ground feature height %d does not match the %s heads (%d)" % (Hg, spec.name,
                                                                                               spec.grd_feat_h))
        scratch_g = torch.empty(6 * Bg * Kg * Wg, dtype=f32, device=dev)
        g: List[torch.Tensor] = [torch.empty((Bg, Wg * h[0].shape[0]), dtype=f32, device=dev) for h in w["heads"]]
        heads = w["heads"]
        ctot = sum(h[0].shape[0] for h in heads)
        self._op("grd_project_tiled_kernel:grd_descriptors|", 2.0 * Bg * Wg * Kg * (6 * Hg + ctot),
                 grd_feat.numel() * grd_feat.element_size() + sum(t.numel() for t in g) * 4,
                 lambda: cabi.grd_descriptors(grd_feat, heads, g, scratch_g))

        # a3 -- aerial cell descriptors: [B,16,16,1280] -> [B,8,8,D]
        fs = _cl(sat_feat, dtype)
        Hs, Ws = fs.shape[1], fs.shape[2]
        D = spec.sat_dim
        x = torch.empty((B, Hs // 2, Ws // 2, D), dtype=dtype, device=dev)
        self._igemm("igemm:cell|", fs, ENCODER_CHANNELS, None, 0, B, Hs, Ws, Hs // 2, Ws // 2, 2, 2, 0, D, dtype,
                    w["cell"], x, 0, D)
        skips = [_cl(multiscale[i], dtype) for i in SKIP_BLOCKS]
        if save is not None:
            save.update(dtype=dtype, B=B, grd_feat=grd_feat, fs=fs, skips=skips, g=g, loc=[], ori=[])

        # The orientation decoder only needs level 1 (score volume + normalised map) and the skips: it runs on a forked side
        # stream, concurrently with levels 2..6 of the localisation decoder (per-operator timing runs them back to back)
        fork = Fork(dev, enabled=self.timer is None and self.concurrent)

        def orientation_decoder():
            # a11 -- orientation decoder (no matching inside; input = [scores_1, normalize(x_1)], models.py:323)
            o = None
            for l in range(6):
                ow = w["ori"][l]
                nm = "ori%d" % (6 - l)
                o_in = o
                if l == 0:
                    o = self._deconv(ow["deconv"], scores_cl, SCORES_CL_PAD, xhat, D, dtype, name=nm)
                else:
                    o = self._deconv(ow["deconv"], o, o.shape[-1], None, 0, dtype, name=nm)
                o_up = o
                if l < 5:
                    o = self._conv3(ow["conv_a"], o, skips[l], dtype, relu=True, name=nm + "a")
                    o_h = o
                    o = self._conv3(ow["conv_b"], o, None, dtype, relu=False, name=nm + "b")
                else:
                    o = self._conv3(ow["conv_a"], o, None, dtype, relu=True, name=nm + "a")
                    o_h = o
                    o = self._conv3(ow["conv_b"], o, None, dtype, relu=False, out_f32=True, name=nm + "b")  # fp32 [B,512,512,2]
                if save is not None:
                    save["ori"].append(dict(inp=o_in, up=o_up, h=o_h))
            Ho, Wo = o.shape[1], o.shape[2]
            ori_ = torch.empty((B, 2, Ho, Wo), dtype=f32, device=dev)
            self._op("ori_normalize_kernel:ori_normalize|", 6.0 * B * Ho * Wo, 2.0 * B * Ho * Wo * (o.element_size() + 4),
                     lambda: cabi.ori_normalize(o, ori_))                                   # a12
            return o, ori_

        o_raw = ori = None
        loc_rolls = loc_roll_indices(spec, self.ori_noise)
        scores_out: List[torch.Tensor] = []
        scores_cl = xhat = None
        logits = None
        for l in range(6):
            _, H, W, C = x.shape
            L = g[l].shape[1]
            if spec.window_len(C, L) != L or L > C:
                raise cabi.CcvpeError("level %d: ground descriptor length %d incompatible with %d aerial channels"
                                      % (l + 1, L, C))
            stride = spec.roll_strides[l]
            if l == 0 and self.ori_noise is not None:
                # full sweep for the orientation decoder, prior-limited subset for the max (models.py:489-511)
                if spec.n_rolls * stride != C:
                    raise cabi.CcvpeError("prior-limited matching needs a full-circle level-1 map")
                rolls = list(range(spec.n_rolls))
                mask = 0
                for i in loc_rolls:
                    mask |= 1 << (i % spec.n_rolls)
            else:
                rolls = loc_rolls
                mask = (1 << len(rolls)) - 1
            R = len(rolls)
            scores = torch.empty((B, R, H, W), dtype=f32, device=dev)
            mx = torch.empty((B, H, W), dtype=f32, device=dev)
            inv = torch.empty((B, H, W), dtype=f32, device=dev)
            if l == 0:
                scores_cl = torch.empty((B, H, W, SCORES_CL_PAD), dtype=dtype, device=dev)
                xhat = torch.empty_like(x)
            scratch = torch.empty(cabi.match_scratch_elems(B, C, R), dtype=f32, device=dev)
            x_in, g_in = x, g[l]
            # algorithmic traffic (SURVEY section 8(d)): read x once, write the score volume + max + 1/norm
            nbytes = x.numel() * x.element_size() + (R + 2) * B * H * W * 4
            mk = "match" if self.timer is None else cabi.match_kernel_name(
                dtype, C, L, spec.window_offset(C, L), [i * stride for i in rolls], SCORES_CL_PAD if l == 0 else 0,
                cabi.BACKEND_SIMT if self.backend == cabi.BACKEND_SIMT else cabi.BACKEND_AUTO)
            self._op(mk + ":match|l%d" % (l + 1), 2.0 * R * L * B * H * W, nbytes, lambda: cabi.match_level(
                x_in, g_in, spec.window_offset(C, L), [i * stride for i in rolls], mask, scores=scores,
                scores_cl=scores_cl if l == 0 else None, max_out=mx, inv_norm=inv,
                xhat=xhat if l == 0 else None, scratch=scratch,
                backend=cabi.BACKEND_SIMT if self.backend == cabi.BACKEND_SIMT else cabi.BACKEND_AUTO))
            scores_out.append(scores)
            if l == 0:
                with fork:
                    o_raw, ori = orientation_decoder()
            lw = w["loc"][l]
            nm = "loc%d" % (6 - l)
            x_level = x
            up = self._deconv(lw["deconv"], x, C, None, 0, dtype, row_scale=inv, row_r1=mx, name=nm)
            if l < 5:
                h = self._conv3(lw["conv_a"], up, skips[l], dtype, relu=True, name=nm + "a")
                x = self._conv3(lw["conv_b"], h, None, dtype, relu=False, name=nm + "b")
            else:
                h = self._conv3(lw["conv_a"], up, None, dtype, relu=True, name=nm + "a")
                logits = self._conv3(lw["conv_b"], h, None, dtype, relu=False, planar_f32=True,
                                     name=nm + "b")                                              # [B,1,512,512]
            if save is not None:
                save["loc"].append(dict(x=x_level, scores=scores, mx=mx, inv=inv, up=up, h=h, mask=mask,
                                        shifts=[i * stride for i in rolls], offset=spec.window_offset(C, L)))

        # a10 -- heatmap
        Hh, Wh = logits.shape[-2:]
        logits_flat = logits.view(B, Hh * Wh)
        heatmap = torch.empty_like(logits)
        sm_scratch = torch.empty(cabi.softmax_scratch_elems(B, Hh * Wh), dtype=f32, device=dev)
        self._op("softmax_finish_kernel:softmax|", 5.0 * B * Hh * Wh, 2.0 * B * Hh * Wh * 4,
                 lambda: cabi.softmax_heatmap(logits_flat, heatmap.view(B, Hh * Wh), sm_scratch))
        side_saved = [t for rec in save["ori"] for t in rec.values()] if save is not None else []
        fork.join(ori, o_raw, *side_saved)
        if save is not None:
            save.update(o_raw=o_raw, scores_cl=scores_cl, xhat=xhat)
        return (logits_flat, heatmap, ori, *scores_out)


@torch.no_grad()
def decode_pose(heatmap: torch.Tensor, ori: torch.Tensor) -> Dict[str, torch.Tensor]:
    """a13 -- device-side replacement of the scripts' NumPy decode (reference train_VIGOR.py:290-326).

    heatmap [B,1,H,W] fp32, ori [B,2,H,W] fp32 (CUDA).  Returns CUDA tensors: idx int64[B], rc int32[B,2] (row, col),
    cs float32[B,2], angle float64[B] (degrees, NaN where invalid), valid uint8[B]."""
    if not heatmap.is_cuda:
        raise cabi.CcvpeError("decode_pose needs CUDA tensors; there is no CPU fallback")
    heatmap = heatmap.contiguous().float()
    ori = ori.contiguous().float()
    B, _, H, W = heatmap.shape
    dev = heatmap.device
    out = dict(idx=torch.empty(B, dtype=torch.int64, device=dev), rc=torch.empty((B, 2), dtype=torch.int32, device=dev),
               cs=torch.empty((B, 2), dtype=torch.float32, device=dev),
               angle=torch.empty(B, dtype=torch.float64, device=dev), valid=torch.empty(B, dtype=torch.uint8, device=dev))
    scratch = torch.empty(cabi.pose_scratch_bytes(B, H * W), dtype=torch.uint8, device=dev)
    with cabi.device_of(heatmap):
        cabi.pose_decode(heatmap, ori, out["idx"], out["rc"], out["cs"], out["angle"], out["valid"], scratch)
    return out


@torch.no_grad()
def decode_hypotheses(heatmap: torch.Tensor, ori: torch.Tensor, k: int, radius: int) -> Dict[str, torch.Tensor]:
    """The k strongest mutually exclusive location modes of each heatmap, in one launch (include/ccvpe_b200.h,
    ccvpe_pose_hypotheses).  A mode is a pixel >= its 8 neighbours; modes are taken highest first (ties: smaller flat
    index), each one claims the disc of `radius` pixels around it, and a mode inside an earlier disc is skipped.

    heatmap [B,1,H,W] fp32, ori [B,2,H,W] fp32 (CUDA).  Returns CUDA tensors: decode_pose's keys per hypothesis -- idx
    int64[B,k], rc int32[B,k,2], cs float32[B,k,2], angle float64[B,k], valid uint8[B,k] -- plus value float32[B,k] (the
    heatmap at the mode), mass float32[B,k] (the heatmap summed over the part of its disc no earlier hypothesis claimed;
    mass[:, 0] is a confidence) and count int32[B].  Slots t >= count[b] hold idx -1 and NaN.  A heatmap holding a NaN
    has count 0.  With k = 1, idx / rc / cs / angle / valid equal decode_pose's on every NaN-free map."""
    if not heatmap.is_cuda:
        raise cabi.CcvpeError("decode_hypotheses needs CUDA tensors; there is no CPU fallback")
    heatmap = heatmap.contiguous().float()
    ori = ori.contiguous().float()
    B = heatmap.shape[0]
    dev = heatmap.device
    out = dict(idx=torch.empty((B, k), dtype=torch.int64, device=dev),
               rc=torch.empty((B, k, 2), dtype=torch.int32, device=dev),
               cs=torch.empty((B, k, 2), dtype=torch.float32, device=dev),
               angle=torch.empty((B, k), dtype=torch.float64, device=dev),
               valid=torch.empty((B, k), dtype=torch.uint8, device=dev),
               value=torch.empty((B, k), dtype=torch.float32, device=dev),
               mass=torch.empty((B, k), dtype=torch.float32, device=dev),
               count=torch.empty(B, dtype=torch.int32, device=dev))
    with cabi.device_of(heatmap):
        cabi.pose_hypotheses(heatmap, ori, k, radius, out["idx"], out["rc"], out["value"], out["mass"], out["cs"],
                             out["angle"], out["valid"], out["count"])
    return out


@torch.no_grad()
def track_step(belief: torch.Tensor, heatmap: torch.Tensor, motion: torch.Tensor, sigma: float,
               epsilon: float = 0.0) -> Dict[str, torch.Tensor]:
    """One step of the sequential location filter (include/ccvpe_b200.h, ccvpe_track_step): warps `belief` by `motion`,
    blurs it with a Gaussian of `sigma` pixels, mixes in `epsilon` of the uniform distribution, multiplies by this frame's
    heatmap and renormalises, updating `belief` in place.

    belief fp32 [B,1,H,W] contiguous (CUDA; start a track with a copy of the first heatmap), heatmap [B,1,H,W] fp32,
    motion float64 [B,6] on the device: the affine data (`models.track_motion`) mapping a pixel centre of this frame's
    crop to a coordinate of the previous frame's.  Returns CUDA tensors evidence float64[B] (the sum Z of prior * heatmap:
    the predictive likelihood of the frame) and reset uint8[B] (1 where Z was not a positive finite number and the belief
    restarted as a copy of the heatmap).  Decode the belief with decode_pose / decode_hypotheses."""
    if not belief.is_cuda:
        raise cabi.CcvpeError("track_step needs CUDA tensors; there is no CPU fallback")
    heatmap = heatmap.contiguous().float()
    B, _, H, W = belief.shape
    dev = belief.device
    out = dict(evidence=torch.empty(B, dtype=torch.float64, device=dev), reset=torch.empty(B, dtype=torch.uint8, device=dev))
    scratch = torch.empty(max(cabi.track_scratch_bytes(B, H, W), 0), dtype=torch.uint8, device=dev)
    with cabi.device_of(belief):
        cabi.track_step(belief, heatmap, motion, sigma, epsilon, out["evidence"], out["reset"], scratch)
    return out
