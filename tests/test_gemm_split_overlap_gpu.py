"""Split-fp16 tcgen05 GEMM with several tiles per CTA on the tile widths whose two accumulators fill TMEM (pair 192 / 256, 1-CTA
144).  At 144 and 192 the epilogue gives the accumulator back before its math and stores, so the MMAs of the next tile run while
the epilogue variant works from its parked copy; large-M launches walk row bands.  Every epilogue variant is checked against
float64 and bit for bit against the same product computed in <= 128-column slices of B, which run the double-buffered 128-wide
kernel and issue the same k-steps per output element."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from roma_b200 import cabi  # noqa: E402
from roma_b200.cabi import call  # noqa: E402
from roma_b200.packing import Split  # noqa: E402

DEV = "cuda"
F32, F16S = cabi.RB_F32, cabi.RB_F16S
VARIANTS = ["bias", "bias_gelu_split_out", "relu", "col_scale_inplace_residual", "alpha", "direct_store", "exp_cosine"]
# (M, N, K): pair 192 (3.2 and 3.8 tiles per cluster), pair 256 (4.3), 1-CTA 144 (3.2 per CTA); ragged M and N tails throughout
SHAPES = [(20000, 569, 569), (12000, 1137, 1137), (20000, 1024, 1024), (60000, 144, 144)]


def pad8(n):
    return (n + 7) // 8 * 8


def rnd(*shape, seed=0, scale=1.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(DEV)


def dev_split(x, rows, cols, ld):
    hi = torch.zeros((rows, ld), dtype=torch.float16, device=DEV)
    lo = torch.zeros((rows, ld), dtype=torch.float16, device=DEV)
    call("romab200_split_f16s", "rb_split_pair_args", x=x, hi=hi, lo=lo, rows=rows, cols=cols, ldx=x.stride(0), ldd=ld)
    return Split(hi, lo)


class Problem:
    def __init__(self, M, N, K, seed=0):
        self.M, self.N, self.K, self.ld = M, N, K, pad8(K)
        A, B = rnd(M, self.ld, seed=seed + 1), rnd(N, self.ld, seed=seed + 2, scale=0.05)
        A[:, K:] = 0
        B[:, K:] = 0
        self.A, self.B = A, B
        self.sa, self.sb = dev_split(A, M, K, self.ld), dev_split(B, N, K, self.ld)
        self.bias, self.gamma = rnd(N, seed=seed + 3), rnd(N, seed=seed + 4)
        self.na, self.nb = A.norm(dim=1).contiguous(), B.norm(dim=1).contiguous()
        self.prod = A[:, :K].double() @ B[:, :K].double().t()
        f32 = A[:, :K] @ B[:, :K].t()
        self.tol = ((f32.double() - self.prod).abs().max() / self.prod.abs().max()).item() + 2.0 ** -20 + 0.5 * (K / 16) * 2.0 ** -24


def out_spec(p, variant):
    """(ldc, output tensor or Split) of a variant, filled with the same start values every time."""
    if variant == "bias_gelu_split_out":
        ldc = pad8(p.N)
        return ldc, Split(torch.full((p.M, ldc), 3.0, dtype=torch.float16, device=DEV), torch.full((p.M, ldc), 3.0, dtype=torch.float16, device=DEV))
    ldc = p.N + 1 if variant == "direct_store" else (p.N + 3) // 4 * 4       # odd fp32 pitch: no TMA store, per-lane direct stores
    if variant == "col_scale_inplace_residual":
        return ldc, rnd(p.M, ldc, seed=9)
    return ldc, torch.full((p.M, ldc), 3.0, device=DEV)


def run(p, variant, C, ldc, n0=0, n=None):
    """C[:, n0:n0+n] = variant(A @ B[n0:n0+n].T) through romab200_gemm (raw pointers for the column slice)."""
    n = p.N - n0 if n is None else n
    boff = n0 * p.ld * 2
    args = dict(A=p.sa.hi, A_lo=p.sa.lo, B=p.sb.hi.data_ptr() + boff, B_lo=p.sb.lo.data_ptr() + boff, M=p.M, N=n, K=p.K, lda=p.ld, ldb=p.ld, ldc=ldc,
                dtype_ab=F16S, batch0=1, batch1=1, ntaps=1, alpha=1.0, backend=cabi.BACKEND_TCGEN05)
    if isinstance(C, Split):
        args.update(C=C.hi.data_ptr() + 2 * n0, C_lo=C.lo.data_ptr() + 2 * n0, dtype_c=F16S)
    else:
        args.update(C=C.data_ptr() + 4 * n0, dtype_c=F32)
    vec = lambda t: t.data_ptr() + 4 * n0
    if variant in ("bias", "bias_gelu_split_out", "relu", "direct_store", "col_scale_inplace_residual"):
        args.update(bias=vec(p.bias))
    if variant == "bias_gelu_split_out":
        args.update(act=cabi.ACT_GELU)
    elif variant == "relu":
        args.update(act=cabi.ACT_RELU)
    elif variant == "col_scale_inplace_residual":
        args.update(col_scale=vec(p.gamma), R=args["C"], ldr=ldc, dtype_r=F32)
    elif variant == "alpha":
        args.update(alpha=0.5)
    elif variant == "exp_cosine":
        args.update(epi=cabi.EPI_COSKERNEL, norm_a=p.na, norm_b=vec(p.nb), eps=1e-6, inv_t=5.0, diag_add=0.0, cos_normalized=0)
    call("romab200_gemm", "rb_gemm_args", **args)


def reference(p, variant, start):
    base = p.prod + p.bias.double()
    if variant == "bias" or variant == "direct_store":
        return base
    if variant == "bias_gelu_split_out":
        return torch.nn.functional.gelu(base)
    if variant == "relu":
        return base.clamp_min(0)
    if variant == "col_scale_inplace_residual":
        return start[:, :p.N].double() + base * p.gamma.double()
    if variant == "alpha":
        return 0.5 * p.prod
    cos = p.prod / (p.na.double()[:, None] * p.nb.double()[None] + 1e-6)
    return ((cos - 1.0) * 5.0).exp()


def values(C, N):
    return (C.join() if isinstance(C, Split) else C)[:, :N].double()


_cache = {}


def problem(M, N, K):
    if (M, N, K) not in _cache:
        _cache.clear()
        _cache[(M, N, K)] = Problem(M, N, K)
    return _cache[(M, N, K)]


@pytest.mark.parametrize("M,N,K", SHAPES)
@pytest.mark.parametrize("variant", VARIANTS)
def test_split_gemm_wide_tiles_epilogues(M, N, K, variant):
    p = problem(M, N, K)
    ldc, C = out_spec(p, variant)
    start = None if isinstance(C, Split) else C.clone()
    run(p, variant, C, ldc)
    _, S = out_spec(p, variant)
    for n0 in range(0, N, 128):
        run(p, variant, S, ldc, n0, min(128, N - n0))
    torch.cuda.synchronize()
    got, ref = values(C, N), reference(p, variant, start)
    if variant == "exp_cosine":
        assert (got - ref).abs().max().item() < 3e-5
    else:
        tol = p.tol + (2.0 ** -21 if isinstance(C, Split) else 0.0)      # the split-pair output adds its own 2^-22 representation
        err = ((got - ref).abs().max() / ref.abs().max()).item()
        assert err <= tol, (err, tol)
    if isinstance(C, Split):
        assert torch.equal(C.hi, S.hi) and torch.equal(C.lo, S.lo)
    else:
        assert torch.equal(C, S)


def test_split_gemm_band_major_beyond_l2():
    """A split A operand of 137 MB (larger than L2) with three 192-wide N tiles: the launch walks row bands."""
    M, N, K = 60000, 569, 569
    p = Problem(M, N, K, seed=20)
    assert 2 * 2 * M * p.ld >= 130e6
    ldc = (N + 3) // 4 * 4
    C, S = torch.full((M, ldc), 3.0, device=DEV), torch.full((M, ldc), 3.0, device=DEV)
    run(p, "bias", C, ldc)
    for n0 in range(0, N, 128):
        run(p, "bias", S, ldc, n0, min(128, N - n0))
    torch.cuda.synchronize()
    ref = p.prod + p.bias.double()
    err = ((C[:, :N].double() - ref).abs().max() / ref.abs().max()).item()
    assert err <= p.tol, (err, p.tol)
    assert torch.equal(C, S)
