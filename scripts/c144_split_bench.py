"""CUDA-event timing of one stride-2 refiner block in the parity mode at the shapes of bench.py (560 -> 864, symmetric pair:
D = 2 maps of 280 x 280 and 432 x 432, C = 144): the fused fp32 / split-fp16 kernel against the depthwise kernel + split
GEMM pair it replaces, with the HBM and FFMA floors of each shape.  The maps (90 / 215 MB) exceed the 126 MB L2 at 432^2;
the blocks ping-pong between two maps as in the engine.

    python scripts/c144_split_bench.py [iters]
"""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from roma_b200 import cabi
from roma_b200.cabi import call
from roma_b200.packing import split_f16s

C = 144
HBM_TBS = 6.5          # measured stream bandwidth of the B200 (DESIGN.md)


def timed(fn, iters):
    for _ in range(3):
        fn()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for _ in range(iters):
        fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) * 1e3 / iters        # us per launch (pair: per block)


def main():
    iters = int(sys.argv[1]) if len(sys.argv) > 1 else 50
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    except OSError:
        q = "nvidia-smi not available"
    print(f"device: {torch.cuda.get_device_name()} | {q}")
    g = torch.Generator().manual_seed(0)
    dwt = (torch.randn(25, C, generator=g) * 0.3).cuda()
    db, pb = torch.randn(C, generator=g).cuda(), torch.randn(C, generator=g).cuda()
    hi, lo = (t.contiguous().cuda() for t in split_f16s(torch.randn(C, C, generator=g) * 0.1))
    for D, H, W in ((2, 280, 280), (2, 432, 432)):
        rows = D * H * W
        d = torch.randn(rows, C, generator=g).cuda()
        t = torch.empty_like(d)
        ts_hi = torch.empty(rows, C, dtype=torch.float16, device="cuda")
        ts_lo = torch.empty_like(ts_hi)

        def dw():
            call("romab200_dwconv5x5_relu", "rb_dwconv_args", **{"in": d}, out=ts_hi, out_lo=ts_lo, ldi=C, ldo=C, weight=dwt, ldw=C, bias=db,
                 batch=D, h=H, w=W, c=C, dtype=cabi.RB_F32)

        def pw():
            call("romab200_gemm", "rb_gemm_args", A=ts_hi, A_lo=ts_lo, B=hi, B_lo=lo, C=d, M=rows, N=C, K=C, lda=C, ldb=C, ldc=C,
                 dtype_ab=cabi.RB_F16S, dtype_c=cabi.RB_F32, batch0=1, batch1=1, ntaps=1, alpha=1.0, bias=pb)

        bufs = [d, t]

        def fused():
            call("romab200_refiner_block_c144", "rb_refiner_block_c144_args", **{"in": bufs[0]}, out=bufs[1], ld=C, dw_weight=dwt, ldw=C,
                 dw_bias=db, pw_weight=hi, pw_weight_lo=lo, ld_pw=C, pw_bias=pb, batch=D, h=H, w=W, c=C, dtype=cabi.RB_F32)
            bufs.reverse()
        t_dw, t_pw = timed(dw, iters), timed(pw, iters)
        t_pair = timed(lambda: (dw(), pw()), iters)
        t_fused = timed(fused, iters)
        map_bytes = rows * C * 4
        hbm_floor = 2 * map_bytes / (HBM_TBS * 1e12) * 1e6
        fma_floor = rows * C * 25 / (148 * 128 * 1.9e9) * 1e6     # 128 fp32 FMA / clk / SM at ~1.9 GHz
        print(f"D={D} {H}x{W}x{C}: dwconv {t_dw:7.1f} us + split GEMM {t_pw:7.1f} us (pair back to back {t_pair:7.1f}) -> fused {t_fused:7.1f} us "
              f"({t_pair / t_fused:.2f}x); floors: HBM {hbm_floor:.1f} us (2 x {map_bytes / 1e6:.0f} MB at {HBM_TBS} TB/s), FFMA {fma_floor:.1f} us; "
              f"fused = {100 * hbm_floor / t_fused:.0f} % of the HBM floor")


if __name__ == "__main__":
    main()
