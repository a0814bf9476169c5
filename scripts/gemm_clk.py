"""Role-time counters of the tcgen05 GEMM kernels (ROMAB200_TC_CLK=1): where the MMA thread / TMA producer / epilogue wait."""
import ctypes, os, sys
os.environ["ROMAB200_TC_CLK"] = "1"
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from roma_b200 import cabi
from roma_b200.cabi import call

lib = cabi.load_library()
dev = "cuda"
NAMES = ["mma wait full", "mma wait tmem_empty", "mma total", "prod0 wait empty", "prod0 total", "epi wait tmem_full", "epi total(incl wait)", "tiles", "kblocks",
         "prod1 wait empty", "prod1 total"]


def pad8(n):
    return (n + 7) // 8 * 8


def run(name, M, N, K, split, act=0, reps=5, f32_out=False):
    """f32_out: fp32 C with ldc = pad8(N) (the refiner pointwise convolutions); otherwise a 16-bit (split: pair) C with ldc = N."""
    lda = pad8(K)
    mk = lambda r, c: torch.randn(r, c, device=dev).to(torch.float16)
    A, Al, B, Bl = mk(M, lda), mk(M, lda), mk(N, lda), mk(N, lda)
    ldc = pad8(N) if f32_out else N
    args = dict(A=A, B=B, M=M, N=N, K=K, lda=lda, ldb=lda, ldc=ldc, ntaps=1, dtype_ab=cabi.RB_F16S if split else cabi.RB_F16, batch0=1, batch1=1,
                alpha=1.0, bias=torch.randn(N, device=dev), act=act)
    if split:
        args.update(A_lo=Al, B_lo=Bl)
    if f32_out:
        args.update(C=torch.empty(M, ldc, device=dev), dtype_c=cabi.RB_F32)
    elif split:
        args.update(C=torch.empty(M, ldc, device=dev, dtype=torch.float16), C_lo=torch.empty(M, ldc, device=dev, dtype=torch.float16), dtype_c=cabi.RB_F16S)
    else:
        args.update(C=torch.empty(M, ldc, device=dev, dtype=torch.float16), dtype_c=cabi.RB_F16)
    for _ in range(2):
        call("romab200_gemm", "rb_gemm_args", **args)
    torch.cuda.synchronize()
    out = (ctypes.c_ulonglong * 16)()
    lib.romab200_debug_tc_clk(out, 1)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        call("romab200_gemm", "rb_gemm_args", **args)
    e.record(); torch.cuda.synchronize()
    lib.romab200_debug_tc_clk(out, 1)
    v = [x / reps for x in out]
    tiles, kb = max(v[7], 1), max(v[8], 1)
    n_mma = 74 if v[9] > 0 else 148        # MMA threads: one per pair or one per CTA (approx., full grid)
    ew = tiles * (2 if v[9] > 0 else 1)        # epilogue-timing warps: warp 2 of every CTA
    print(f"    epilogue phases per tile [cycles] (EPI={os.environ.get('ROMAB200_GEMM_EPI', '1')}): pre(vectors+barriers) {v[11] / ew:.0f}, wait acc {v[5] / ew:.0f}, "
          f"tmem ld {v[12] / ew:.0f}, math {v[13] / ew:.0f}, store {v[14] / ew:.0f}")
    print(f"{name}: {s.elapsed_time(e) / reps * 1e3:.1f} us; per k-block [cycles]: mma total {v[2] / kb:.0f}, wait full {v[0] / kb:.0f}, wait tmem {v[1] / kb:.0f}; "
          f"prod0 wait empty {v[3] / kb:.0f} of {v[4] / kb:.0f}; per tile: epi total {v[6] / tiles:.0f}; tiles {tiles:.0f} kblocks {kb:.0f}", flush=True)
    print(f"    MMA thread per tile [cycles]: total {v[2] / tiles:.0f}, wait tmem_empty {v[1] / tiles:.0f} ({100 * v[1] / max(v[2], 1):.1f} %), "
          f"wait full {v[0] / tiles:.0f}", flush=True)


print("device:", torch.cuda.get_device_name(), "| PAIR =", os.environ.get("ROMAB200_GEMM_PAIR", "1"), "| BN =", os.environ.get("ROMAB200_GEMM_BN", "auto"))
for split in (True, False):
    t = "split" if split else "fp16 "
    run(f"{t} fc1 3202x4096x1024 gelu", 3202, 4096, 1024, split, cabi.ACT_GELU)
    run(f"{t} qkv 3202x3072x1024", 3202, 3072, 1024, split)
    run(f"{t} fc2->f32 3202x1024x4096", 3202, 1024, 4096, split)
# refiner pointwise convolutions of the parity mode: fp32 out with bias, ldc = pad8(N)
for M, N, K, what in ((93312, 569, 569, "stride 4 @864"), (23328, 1137, 1137, "stride 8 @864"), (39200, 569, 569, "stride 4 @560")):
    run(f"split refiner pw {M}x{N}x{K} ({what}) ->f32", M, N, K, True, f32_out=True)
