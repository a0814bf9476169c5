"""Fused stride-2 refiner block on fp32 maps (romab200_refiner_block_c144 with dtype RB_F32): depthwise 5x5 + ReLU on the
CUDA cores feeding the split-fp16 tcgen05 pointwise GEMM in one kernel.  It does the arithmetic of the un-fused pair
(romab200_dwconv5x5_relu into an RB_F16S pair, then the split romab200_gemm with the bias), so its output must be the
same bits; a float64 reference bounds both at the split-fp32 level."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from roma_b200 import cabi  # noqa: E402
from roma_b200.cabi import call  # noqa: E402
from roma_b200.packing import split_f16s  # noqa: E402

DEV = "cuda"
C = 144


def rnd(*shape, seed=0, scale=1.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return torch.randn(*shape, generator=g) * scale


def block_inputs(B, H, W, scale):
    x = rnd(B, H, W, C, seed=1, scale=scale)
    dw, db = rnd(C, 1, 5, 5, seed=2, scale=0.3), rnd(C, seed=3, scale=scale)
    pw, pb = rnd(C, C, seed=4, scale=0.1), rnd(C, seed=5, scale=scale)
    return x, dw, db, pw, pb


def run_both(x, dw, db, pw, pb):
    B, H, W, _ = x.shape
    rows = B * H * W
    xi = x.to(DEV).contiguous()
    dwt = dw.reshape(C, 25).t().contiguous().to(DEV)
    db_d, pb_d = db.to(DEV), pb.to(DEV)
    hi, lo = (t.contiguous().to(DEV) for t in split_f16s(pw))
    # un-fused: depthwise kernel -> RB_F16S pair in memory -> split GEMM with the bias
    ts_hi = torch.full((rows, C), 7.0, dtype=torch.float16, device=DEV)
    ts_lo = torch.full((rows, C), 7.0, dtype=torch.float16, device=DEV)
    call("romab200_dwconv5x5_relu", "rb_dwconv_args", **{"in": xi}, out=ts_hi, out_lo=ts_lo, ldi=C, ldo=C, weight=dwt, ldw=C, bias=db_d,
         batch=B, h=H, w=W, c=C, dtype=cabi.RB_F32)
    ref = torch.full((B, H, W, C), 7.0, device=DEV)
    call("romab200_gemm", "rb_gemm_args", A=ts_hi, A_lo=ts_lo, B=hi, B_lo=lo, C=ref, M=rows, N=C, K=C, lda=C, ldb=C, ldc=C,
         dtype_ab=cabi.RB_F16S, dtype_c=cabi.RB_F32, batch0=1, batch1=1, ntaps=1, alpha=1.0, bias=pb_d)
    # fused
    out = torch.full((B, H, W, C), 7.0, device=DEV)
    call("romab200_refiner_block_c144", "rb_refiner_block_c144_args", **{"in": xi}, out=out, ld=C, dw_weight=dwt, ldw=C, dw_bias=db_d,
         pw_weight=hi, pw_weight_lo=lo, ld_pw=C, pw_bias=pb_d, batch=B, h=H, w=W, c=C, dtype=cabi.RB_F32)
    torch.cuda.synchronize()
    return out, ref


@pytest.mark.parametrize("B,H,W,scale", [(1, 8, 16, 1.0), (2, 37, 50, 1.0), (1, 21, 35, 1.0), (2, 13, 9, 1e-3), (2, 70, 70, 1e-3),
                                         (2, 432, 432, 1.0)])
def test_fused_split_block_matches_unfused_bitwise(B, H, W, scale):
    """Ragged tiles (H, W not multiples of 8 / 16), B = 1 and 2, small magnitudes (the lo plane carries the low bits) and the
    432 x 432 x 2 map of the upsample pass."""
    x, dw, db, pw, pb = block_inputs(B, H, W, scale)
    out, ref = run_both(x, dw, db, pw, pb)
    diff = (out - ref).abs().max().item()
    assert diff == 0.0, f"fused vs un-fused: max |diff| = {diff:.3e}"
    assert torch.isfinite(out).all()


@pytest.mark.parametrize("B,H,W,scale", [(2, 37, 50, 1.0), (1, 24, 40, 1e-3)])
def test_fused_split_block_vs_float64(B, H, W, scale):
    """Split-fp32 accuracy: the depthwise stage is fp32 FMA, the pointwise operands carry 22 significand bits."""
    x, dw, db, pw, pb = block_inputs(B, H, W, scale)
    out, _ = run_both(x, dw, db, pw, pb)
    mid = F.relu(F.conv2d(x.permute(0, 3, 1, 2).double(), dw.double(), db.double(), padding=2, groups=C))
    ref = torch.einsum("bchw,oc->bhwo", mid, pw.double()) + pb.double()
    err = ((out.double().cpu() - ref).abs().max() / ref.abs().max()).item()
    assert err < 1e-5, err


def test_parity_match_fused_equals_unfused():
    """One small symmetric match() in the parity mode with the fused stride-2 blocks and with the un-fused pair: same bits."""
    from roma_b200 import roma_outdoor, synthetic
    mw, dw = synthetic.make_weights(0)
    A, B, Ah, Bh = synthetic.make_pair(1, 112, 168, seed=1)
    outs = []
    for fused in (True, False):
        model = roma_outdoor("cuda:0", weights=mw, dinov2_weights=dw, coarse_res=112, upsample_res=168, amp_dtype=torch.float32)
        model.engine.fused_c144_f32 = fused
        warp, cert = model.match(A.cuda(), B.cuda(), im_A_high_res=Ah.cuda(), im_B_high_res=Bh.cuda())
        torch.cuda.synchronize()
        outs.append((warp.cpu(), cert.cpu()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
