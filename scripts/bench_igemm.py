"""Micro-benchmark of one implicit-GEMM shape through the C ABI (development tool; inputs > L2 or L2 flushed).

    python scripts/bench_igemm.py conv B c0 c1 cout H [reps]      # 3x3 conv, HxH map
    python scripts/bench_igemm.py deconv B C cout H [reps]        # k2 s2 transposed conv with row-scale + rank-1
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ccvpe_b200 import cabi  # noqa: E402


def main():
    kind = sys.argv[1]
    dev = torch.device("cuda")
    bf = torch.bfloat16
    d = cabi.IgemmDesc()
    if kind == "conv":
        B, c0, c1, cout, H = map(int, sys.argv[2:7])
        reps = int(sys.argv[7]) if len(sys.argv) > 7 else 10
        a0 = torch.randn(B, H, H, c0, device=dev, dtype=bf)
        a1 = torch.randn(B, H, H, c1, device=dev, dtype=bf) if c1 else None
        W = torch.randn(cout, c0 + c1, 3, 3, device=dev) * 0.05
        w_nk = cabi.w_nk_layout(W.permute(0, 2, 3, 1).reshape(cout, 9, c0 + c1), [c0, c1] if c1 else [c0])
        out = torch.empty(B, H, H, cout, device=dev, dtype=bf)
        bias = torch.randn(cout, device=dev)
        d.a0, d.a1, d.c0, d.c1, d.ld0, d.ld1 = a0.data_ptr(), (a1.data_ptr() if c1 else None), c0, c1, c0, c1
        d.B, d.Hin, d.Win, d.Hout, d.Wout = B, H, H, H, H
        d.stride, d.kh, d.kw, d.pad, d.N = 1, 3, 3, 1, cout
        d.out_mode, d.ldo = 0, cout
        flops = 2.0 * B * H * H * cout * 9 * (c0 + c1)
        nbytes = (a0.numel() + (a1.numel() if c1 else 0) + out.numel()) * 2
    else:
        B, C, cout, H = map(int, sys.argv[2:6])
        reps = int(sys.argv[6]) if len(sys.argv) > 6 else 10
        a0 = torch.randn(B, H, H, C, device=dev, dtype=bf)
        W = torch.randn(C, cout, 2, 2, device=dev) * 0.05
        w_nk = cabi.w_nk_layout(W.permute(2, 3, 1, 0).reshape(4 * cout, 1, C), [C])
        out = torch.empty(B, 2 * H, 2 * H, cout, device=dev, dtype=bf)
        bias = torch.randn(4 * cout, device=dev)
        rs = torch.rand(B * H * H, device=dev)
        r1 = torch.rand(B * H * H, device=dev)
        r1w = torch.randn(4 * cout, device=dev)
        d.a0, d.a1, d.c0, d.c1, d.ld0, d.ld1 = a0.data_ptr(), None, C, 0, C, 0
        d.B, d.Hin, d.Win, d.Hout, d.Wout = B, H, H, H, H
        d.stride, d.kh, d.kw, d.pad, d.N = 1, 1, 1, 0, 4 * cout
        d.row_scale, d.row_r1, d.r1_w = rs.data_ptr(), r1.data_ptr(), r1w.data_ptr()
        d.out_mode, d.ldo = 1, cout
        flops = 2.0 * B * H * H * 4 * cout * C
        nbytes = (a0.numel() + out.numel()) * 2
    d.dtype, d.out_dtype, d.w_kn, d.w_nk, d.bias = cabi.BF16, cabi.BF16, None, w_nk.data_ptr(), bias.data_ptr()
    d.out, d.backend = out.data_ptr(), cabi.BACKEND_TCGEN05
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    for _ in range(3):
        cabi.igemm(d)
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        cabi.igemm(d)
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    best = min(ms)
    print("%s %s: %.4f ms  %.1f TFLOP/s  %.1f GB/s (algorithmic)" % (kind, sys.argv[2:], best, flops / best / 1e9,
                                                                  nbytes / best / 1e6))


if __name__ == "__main__":
    main()
