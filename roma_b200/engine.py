"""Device pipeline of RoMa's dense matcher: orchestrates the libromab200 kernels.

One `Engine` owns the packed weights, the per-resolution constants and a cache of activation buffers,
and enqueues the whole of `forward_symmetric` / `forward` (`romatch/models/matcher.py:631-670`) plus the
`match()` epilogue on the current CUDA stream through the C ABI.  PyTorch is used for device memory
(`torch.empty/zeros`) and streams only; every arithmetic step is one of our kernels.

Precision regimes (`precision=`):
  "fp32"        parity mode on the tensor cores: activations stay fp32 in HBM, every GEMM operand is carried as an
                RB_F16S pair (fp16 hi plane + 2^11-scaled fp16 lo plane, 22 significand bits) and contracted by
                three tcgen05 MMAs per k-step with fp32 accumulation in TMEM (gemm_tc.cu, SPLIT variant) — fp32-class
                results, comparable to the reference's CPU fp32 path at the 1e-4 level
                (tests/test_e2e_gpu.py::test_match_full_vs_reference_golden);
  "fp32_simt"   the same arithmetic regime with CUDA-core FFMA GEMMs (gemm_simt.cu): the slow cross-check of "fp32";
  "fp16"/"bf16" fast mode, mirrors the reference's CUDA autocast regime (`utils.py:639-653`): 16-bit GEMM
                operands on the tcgen05 tensor pipe with fp32 accumulation, fp32 residual stream,
                LayerNorm, softmax statistics, GP solve, local-correlation accumulation, heads and
                flow/certainty state.

Data layout: channels-last everywhere.  VGG maps carry a 1-pixel zero border ([E, H+2, W+2, C]) so that a
3x3 convolution is a 9-tap shifted-row GEMM over the flattened padded grid.  Flow and certainty travel
together as a 3-channel fp32 state map [D, h, w, 3].
"""
from __future__ import annotations

import math
import os
from contextlib import contextmanager
from typing import Dict, Optional, Tuple

import torch
import torch.nn.functional as F

from . import arch, cabi
from .cabi import call
from .packing import PackedWeights, Split, pad8

PRECISIONS = {"fp32": torch.float32, "fp32_simt": torch.float32, "fp16": torch.float16, "bf16": torch.bfloat16}
F16S = cabi.RB_F16S


class Engine:
    # parity mode: stride-2 refiner blocks as one fused DW + split-fp16 tcgen05-PW kernel (ROMAB200_FUSED_C144_F32=0: the
    # un-fused depthwise kernel + split GEMM pair, which computes the same bits)
    fused_c144_f32 = os.environ.get("ROMAB200_FUSED_C144_F32", "1") != "0"

    def __init__(self, matcher_sd, dino_sd, device, precision: str = "fp32"):
        if precision not in PRECISIONS:
            raise ValueError(f"precision must be one of {list(PRECISIONS)}")
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("roma_b200 runs on a CUDA device only (there is no CPU fallback); "
                               f"got device={device!r}")
        cabi.load_library()
        self.precision = precision
        self.dtype = PRECISIONS[precision]
        self.dt = cabi.DTYPE_CODE[self.dtype]
        self.split = precision == "fp32"         # fp32-class GEMMs on tcgen05 from RB_F16S operand pairs
        self._lane = "main"                      # scratch buffers are per stream ("main" / "side")
        with torch.cuda.device(self.device):
            self.w = PackedWeights(matcher_sd, dino_sd, self.device, self.dtype, split=self.split)
        self._buf: Dict[tuple, torch.Tensor] = {}
        self.generation = 0
        self._const: Dict[tuple, torch.Tensor] = {}
        self.debug: Optional[dict] = None        # set to {} to keep stage tensors (tests)
        self.use_flash_attn = True               # fused tcgen05 attention in the 16-bit modes (else QK^T / softmax / PV GEMMs)
        self.gp_algo = 2 if precision == "fp32_simt" else 3   # 3: 128-wide blocks factored in shared memory + explicit block inverses, the
                                                 # K=128 GEMMs (13 dependent steps) on the tensor cores as split-fp16 pairs; 2: the same with
                                                 # CUDA-core GEMMs; 0: 32-wide launch chain (50 steps); 1: one cooperative persistent kernel.
        self.overlap_cnn = True                  # VGG/proj branch on a side stream, overlapping ViT / GP / decoder
        self.gp_tensor_core = True               # all-pairs CosKernel on tcgen05 (split-fp16 operands) in the 16-bit modes
        self.fused_c144 = True                   # stride-2 refiner blocks as one fused DW + tcgen05-PW kernel
        self.lc_table16 = os.environ.get("ROMAB200_LC_TABLE16", "1") != "0"   # parity mode: stride-16 local correlation gathered from an all-pairs tensor-core table
        self.side_ctas = int(os.environ.get("ROMAB200_SIDE_CTAS", "0"))   # persistent-grid cap of the side stream's GEMMs (0: none)
        self.kde_symmetric = os.environ.get("ROMAB200_KDE_SYM", "1") != "0"   # sample(): KDE over the upper triangle of the pair matrix
        self.lc_tile_radii = (2,)                # fp32 maps: window radii whose prologue also runs the tile-cooperative pass (measured: wins on coherent
                                                 # flow at r = 2, ties with the per-pixel kernel's L1 hits at r = 3; r = 7 uses the table above)
        self.fused_small_f32 = True              # fp32 modes: stride-1 (C = 24) refiner blocks as one fused fp32 CUDA-core kernel
        self._side = None
        self.profile: Optional[dict] = None      # set to {} to collect CUDA-event timings per stage (bench.py)
        self.gemm_profile: Optional[list] = None  # set to [] to time every GEMM launch: (backend, flops, start, end, shape, epilogue)

    @contextmanager
    def stage(self, name):
        """CUDA-event bracket on the launch stream around one stage of the pipeline (no-op unless profiling)."""
        if self.profile is None:
            yield
            return
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        yield
        end.record()
        self.profile.setdefault(name, []).append((start, end))

    # ------------------------------------------------------------------ buffers and constants
    def buf(self, name, shape, dtype=None, zero=False):
        dtype = dtype or self.dtype
        key = (name, tuple(shape), dtype)
        t = self._buf.get(key)
        if t is None:
            t = (torch.zeros if zero else torch.empty)(tuple(shape), dtype=dtype, device=self.device)
            self._buf[key] = t
        return t

    def sbuf(self, name, shape, zero=False) -> Split:
        """A cached RB_F16S buffer: two fp16 planes of `shape`."""
        return Split(self.buf(name + ".hi", shape, torch.float16, zero), self.buf(name + ".lo", shape, torch.float16, zero))

    def free_buffers(self):
        self._buf.clear()
        self.generation += 1       # captured CUDA graphs hold raw pointers into these buffers: the matcher drops them

    def const(self, key, make):
        t = self._const.get(key)
        if t is None:
            t = make().to(self.device)
            self._const[key] = t
        return t

    def grid_axis(self, n):
        """linspace(-1+1/n, 1-1/n, n): pixel-centre coordinates (matcher.py:365-377)."""
        return self.const(("grid", n), lambda: torch.linspace(-1 + 1 / n, 1 - 1 / n, n))

    def window_axis(self, r, n):
        """linspace(-2r/n, 2r/n, 2r+1): local-correlation window offsets (local_correlation.py:93-103)."""
        return self.const(("win", r, n), lambda: torch.linspace(-2 * r / n, 2 * r / n, 2 * r + 1))

    def pos_embed(self, hp, wp):
        """DINOv2 positional embedding resized exactly as `interpolate_pos_encoding` does (dinov2.py:166-190):
        bicubic with scale_factor=(hp+0.1)/37 (NOT size=), computed once per resolution on the host."""
        def make():
            pe = self.w.vit_pos_embed
            n = pe.shape[1] - 1
            side = int(math.sqrt(n))
            if hp * wp == n and hp == wp:
                return pe[0].clone()
            grid = pe[:, 1:].reshape(1, side, side, -1).permute(0, 3, 1, 2)
            grid = F.interpolate(grid, scale_factor=((hp + 0.1) / side, (wp + 0.1) / side), mode="bicubic")
            assert grid.shape[-2:] == (hp, wp)
            return torch.cat((pe[0, :1], grid.permute(0, 2, 3, 1).reshape(hp * wp, -1)), dim=0).contiguous()
        return self.const(("pos", hp, wp), make)

    def gp_basis_t(self, h, w):
        """F^T [512, h*w]: cos(8*pi*pos_conv(pixel-centre grid)) (matcher.py:264-289), a per-resolution constant."""
        def make():
            ys = torch.linspace(-1 + 1 / h, 1 - 1 / h, h)
            xs = torch.linspace(-1 + 1 / w, 1 - 1 / w, w)
            gy, gx = torch.meshgrid(ys, xs, indexing="ij")
            coords = torch.stack((gx, gy))[None]
            f = torch.cos(8 * math.pi * F.conv2d(coords, self.w.gp_pos_w, self.w.gp_pos_b))
            return f[0].reshape(arch.GP_DIM, h * w).contiguous()
        return self.const(("gpbasis", h, w), make)

    # ------------------------------------------------------------------ kernel wrappers
    def split_pair(self, x, rows, cols, ld, name=None, row_norm=None) -> Split:
        """fp32 matrix [rows, cols] (pitch ld) -> RB_F16S planes of the same pitch (a per-stream scratch pair unless named)."""
        ldd = pad8(ld)
        out = self.sbuf(name or f"split.{self._lane}.{rows * ldd}", (rows * ldd,))
        call("romab200_split_f16s", "rb_split_pair_args", x=x, hi=out.hi, lo=out.lo, rows=rows, cols=cols, ldx=ld, ldd=ldd, row_norm=row_norm)
        return out

    def gemm(self, A, B, C, M, N, K, lda, ldb, ldc, dtype_ab=None, dtype_c=None, **kw):
        args = dict(M=M, N=N, K=K, lda=lda, ldb=ldb, ldc=ldc, batch0=1, batch1=1, ntaps=1, alpha=1.0)
        if self._lane == "side" and self.side_ctas:
            args["max_ctas"] = self.side_ctas        # the CNN branch leaves SMs to the main stream's chain of short kernels (GP solve)
        args.update(kw)
        if (self.split and dtype_ab is None) or isinstance(A, Split):
            # parity mode (and the GP block of every tensor-core mode): operands as RB_F16S pairs.  Activations that no kernel wrote in that format are split here.
            if not isinstance(A, Split):
                assert args["batch0"] * args["batch1"] == 1 and lda % 8 == 0, "batched fp32 operands are split by the caller"
                A = self.split_pair(A, args.get("a_rows") or M, K // args["ntaps"], lda)
            if not isinstance(B, Split):
                assert args["batch0"] * args["batch1"] == 1 and ldb % 8 == 0
                tb = args.get("trans_b", 0)
                B = self.split_pair(B, K if tb else N, N if tb else K, ldb, name=f"splitb.{self._lane}.{(K if tb else N) * ldb}")
            dtype_ab = F16S
            args.update(A=A.hi, A_lo=A.lo, B=B.hi, B_lo=B.lo)
            if isinstance(C, Split):
                args.update(C=C.hi, C_lo=C.lo)
                dtype_c = F16S
            else:
                args.update(C=C)
        else:
            args.update(A=A, B=B, C=C)
        args["dtype_ab"] = self.dt if dtype_ab is None else dtype_ab
        args["dtype_c"] = self.dt if dtype_c is None else dtype_c
        if self.gemm_profile is None:
            call("romab200_gemm", "rb_gemm_args", **args)
            return
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        call("romab200_gemm", "rb_gemm_args", **args)
        end.record()
        flops = 2.0 * M * N * K * args["batch0"] * args["batch1"]
        backend = {cabi.RB_F32: "simt", F16S: "tcgen05-split"}.get(args["dtype_ab"], "tcgen05")
        self.gemm_profile.append((backend, flops, start, end, (M, N, K, args["batch0"] * args["batch1"]), args.get("epi", cabi.EPI_LINEAR)))

    def layernorm(self, x, y, gb, rows, cols, eps, dtype_y=None):
        if isinstance(y, Split):
            call("romab200_layernorm", "rb_layernorm_args", x=x, y=y.hi, y_lo=y.lo, gamma=gb[0], beta=gb[1], rows=rows, cols=cols,
                 ldx=cols, ldy=cols, dtype_x=cabi.RB_F32, dtype_y=F16S, eps=eps)
            return
        call("romab200_layernorm", "rb_layernorm_args", x=x, y=y, gamma=gb[0], beta=gb[1], rows=rows, cols=cols,
             ldx=cols, ldy=cols, dtype_x=cabi.RB_F32, dtype_y=self.dt if dtype_y is None else dtype_y, eps=eps)

    def copy2d(self, src, dst, rows, cols, lds, ldd, ds, dd):
        call("romab200_copy2d", "rb_copy2d_args", src=src, dst=dst, rows=rows, cols=cols, lds=lds, ldd=ldd,
             dtype_src=ds, dtype_dst=dd)

    # ------------------------------------------------------------------ VGG19-BN (encoders.py:17-27)
    def vgg(self, image: torch.Tensor, tag: str):
        """image [E,3,H,W] fp32 -> {s: zero-padded channels-last tap [E, H/s+2, W/s+2, C_s]} for s in 1,2,4,8.
        In the parity mode the maps are RB_F16S pairs (every consumer is a GEMM or the max-pool)."""
        E, _, H, W = image.shape
        taps = {}
        layers = self.w.vgg
        h, w = H, W
        mk = (lambda name, shape: self.sbuf(name, shape, zero=True)) if self.split else (lambda name, shape: self.buf(name, shape, zero=True))
        cur = mk(f"vgg{tag}.s1.in", (E, h + 2, w + 2, 64))
        if self.split:
            call("romab200_conv3x3_first", "rb_conv_first_args", image=image, out=cur.hi, out_lo=cur.lo, weight=layers[0]["w"], bias=layers[0]["b"],
                 batch=E, height=h, width=w, cout=64, dtype_out=F16S)
        else:
            call("romab200_conv3x3_first", "rb_conv_first_args", image=image, out=cur, weight=layers[0]["w"], bias=layers[0]["b"],
                 batch=E, height=h, width=w, cout=64, dtype_out=self.dt)
        li, scale = 1, 1
        for nconv in (1, 2, 4, 4):                              # convs left in each stage after conv0
            for j in range(nconv):
                L = layers[li]
                li += 1
                nxt = mk(f"vgg{tag}.s{scale}.p{j % 2}", (E, h + 2, w + 2, L["cout"]))
                rows = E * (h + 2) * (w + 2)
                taps_rows = [(ky - 1) * (w + 2) + (kx - 1) for ky in range(3) for kx in range(3)]
                self.gemm(cur, L["w"], nxt, rows, L["cout"], 9 * L["cin"], L["cin"], 9 * L["cin"], L["cout"],
                          ntaps=9, tap_rows=taps_rows, a_rows=rows, bias=L["b"], act=cabi.ACT_RELU,
                          rowmap=cabi.ROWMAP_PAD_KEEP, pad_h=h + 2, pad_w=w + 2)
                cur = nxt
            taps[scale] = (cur, h, w)
            if scale == 8:
                break
            c = layers[li - 1]["cout"]
            pooled = mk(f"vgg{tag}.s{scale * 2}.in", (E, h // 2 + 2, w // 2 + 2, c))
            if self.split:
                call("romab200_maxpool2x2_padded", "rb_maxpool_args", **{"in": cur.hi}, in_lo=cur.lo, out=pooled.hi, out_lo=pooled.lo,
                     batch=E, height=h, width=w, channels=c, dtype=F16S)
            else:
                call("romab200_maxpool2x2_padded", "rb_maxpool_args", **{"in": cur}, out=pooled, batch=E, height=h, width=w,
                     channels=c, dtype=self.dt)
            cur, h, w, scale = pooled, h // 2, w // 2, scale * 2
        return taps

    # ------------------------------------------------------------------ transformer blocks
    def attention(self, qkv, out, Bn, N, heads, dim, tag):
        """softmax(q k^T / sqrt(d)) v per head (F.scaled_dot_product_attention, attention.py:50-63).
        qkv [Bn, N, 3*dim] (q|k|v, heads contiguous inside each) -> out [Bn, N, dim]."""
        d = dim // heads
        if self.dtype != torch.float32 and self.use_flash_attn:
            with self.stage(f"  attn.{tag}"):
                call("romab200_flash_attn", "rb_flash_attn_args", qkv=qkv, out=out, ld_qkv=3 * dim, ld_out=dim, batch=Bn, n_tokens=N,
                     heads=heads, head_dim=d, dtype=self.dt)
            return
        npad = pad8(N)
        ld = 3 * dim
        if self.split and d == 64 and self.use_flash_attn:
            # parity mode, ViT heads: fused split-fp16 attention (three MMAs per k-step for QK^T and for PV), no score traffic
            with self.stage(f"  attn.{tag}"):
                call("romab200_flash_attn", "rb_flash_attn_args", qkv=qkv.hi, qkv_lo=qkv.lo, out=out.hi, out_lo=out.lo, ld_qkv=ld, ld_out=dim,
                     batch=Bn, n_tokens=N, heads=heads, head_dim=d, dtype=F16S)
            return
        if self.split:
            # parity mode: q, k, v, the probabilities and the result are RB_F16S pairs; scores are fp32.  The 1/sqrt(d) scale
            # rides on the QK^T epilogue like below.
            S = self.buf(f"attn.scores.{tag}", (Bn, heads, N, npad), dtype=torch.float32)
            P = self.sbuf(f"attn.probs.{tag}", (Bn, heads, N, npad))
            q, k, v = qkv, qkv.at(dim), qkv.at(2 * dim)
            with self.stage(f"  attn.{tag}"):
                self.gemm(q, k, S, N, N, d, ld, ld, npad, batch0=Bn, batch1=heads, alpha=1.0 / math.sqrt(d), dtype_c=cabi.RB_F32,
                          sa0=N * ld, sa1=d, sb0=N * ld, sb1=d, sc0=heads * N * npad, sc1=N * npad)
                call("romab200_softmax_rows", "rb_softmax_args", s=S, rows=Bn * heads * N, cols=N, lds=npad, dtype=cabi.RB_F32, scale=1.0,
                     out_hi=P.hi, out_lo=P.lo, ldo=npad)
                self.gemm(P, v, out, N, d, N, npad, ld, dim, trans_b=1, batch0=Bn, batch1=heads,
                          sa0=heads * N * npad, sa1=N * npad, sb0=N * ld, sb1=d, sc0=N * dim, sc1=d)
            return
        sdt = self.dtype
        S = self.buf(f"attn.scores.{tag}", (Bn, heads, N, npad), dtype=sdt)
        es = qkv.element_size()
        q_ptr, k_ptr, v_ptr = qkv.data_ptr(), qkv.data_ptr() + dim * es, qkv.data_ptr() + 2 * dim * es
        # the 1/sqrt(d) scale rides on the QK^T epilogue so that 16-bit scores cannot overflow
        with self.stage(f"  attn.{tag}"):
            self.gemm(q_ptr, k_ptr, S, N, N, d, ld, ld, npad, batch0=Bn, batch1=heads, alpha=1.0 / math.sqrt(d),
                      sa0=N * ld, sa1=d, sb0=N * ld, sb1=d, sc0=heads * N * npad, sc1=N * npad)
            call("romab200_softmax_rows", "rb_softmax_args", s=S, rows=Bn * heads * N, cols=N, lds=npad, dtype=self.dt, scale=1.0)
            self.gemm(S, v_ptr, out, N, d, N, npad, ld, dim, trans_b=1, batch0=Bn, batch1=heads,
                      sa0=heads * N * npad, sa1=N * npad, sb0=N * ld, sb1=d, sc0=N * dim, sc1=d)

    def block(self, x, blk, Bn, N, dim, heads, mlp, eps, tag):
        """pre-LN transformer block on the fp32 residual stream x [Bn*N, dim] (block.py:82-107)."""
        rows = Bn * N
        mk = self.sbuf if self.split else self.buf       # parity mode: every GEMM operand of the block is an RB_F16S pair
        xn = mk(f"blk.xn.{tag}", (rows, dim))
        qkv = mk(f"blk.qkv.{tag}", (rows, 3 * dim))
        att = mk(f"blk.att.{tag}", (rows, dim))
        hid = mk(f"blk.hid.{tag}", (rows, mlp))
        self.layernorm(x, xn, blk["ln1"], rows, dim, eps)
        self.gemm(xn, blk["qkv_w"], qkv, rows, 3 * dim, dim, dim, dim, 3 * dim, bias=blk["qkv_b"])
        self.attention(qkv, att, Bn, N, heads, dim, tag)
        self.gemm(att, blk["proj_w"], x, rows, dim, dim, dim, dim, dim, dtype_c=cabi.RB_F32, bias=blk["proj_b"],
                  col_scale=blk["ls1"], R=x, ldr=dim, dtype_r=cabi.RB_F32)
        self.layernorm(x, xn, blk["ln2"], rows, dim, eps)
        self.gemm(xn, blk["fc1_w"], hid, rows, mlp, dim, dim, dim, mlp, bias=blk["fc1_b"], act=cabi.ACT_GELU)
        self.gemm(hid, blk["fc2_w"], x, rows, dim, mlp, mlp, mlp, dim, dtype_c=cabi.RB_F32, bias=blk["fc2_b"],
                  col_scale=blk["ls2"], R=x, ldr=dim, dtype_r=cabi.RB_F32)

    # ------------------------------------------------------------------ DINOv2 ViT-L/14 (encoders.py:60-67)
    def dinov2(self, image: torch.Tensor):
        """image [E,3,H,W] fp32 -> patch tokens [E, hp*wp, 1024] in the compute dtype (channels-last stride-14 map)."""
        E, _, H, W = image.shape
        hp, wp = H // arch.VIT_PATCH, W // arch.VIT_PATCH
        npatch, dim = hp * wp, arch.VIT_DIM
        N = npatch + 1
        kp = self.w.vit_patch_w.shape[1]
        cols = self.buf("vit.im2col", (E * npatch, kp), zero=True)
        call("romab200_im2col_patch", "rb_im2col_args", image=image, out=cols, batch=E, height=H, width=W,
             patch=arch.VIT_PATCH, ldo=kp, dtype_out=self.dt)
        patch = self.buf("vit.patch", (E * npatch, dim), dtype=torch.float32)
        self.gemm(cols, self.w.vit_patch_w, patch, E * npatch, dim, 3 * arch.VIT_PATCH ** 2, kp, kp, dim,
                  dtype_c=cabi.RB_F32, bias=self.w.vit_patch_b)
        x = self.buf("vit.x", (E * N, dim), dtype=torch.float32)
        call("romab200_assemble_tokens", "rb_tokens_args", patch=patch, cls=self.w.vit_cls, pos=self.pos_embed(hp, wp),
             tokens=x, batch=E, npatch=npatch, dim=dim)
        for blk in self.w.vit:
            self.block(x, blk, E, N, dim, arch.VIT_HEADS, arch.VIT_MLP, arch.VIT_LN_EPS, "vit")
        out = self.buf("vit.out", (E * N, dim))
        self.layernorm(x, out, self.w.vit_norm, E * N, dim, arch.VIT_LN_EPS)
        feats = self.buf("vit.feat16", (E, npatch, dim))
        # drop the cls token: rows 1..N of every image
        for e in range(E):
            self.copy2d(out.data_ptr() + (e * N + 1) * dim * out.element_size(), feats.data_ptr() + e * npatch * dim * feats.element_size(),
                        npatch, dim, dim, dim, self.dt, self.dt)
        return feats, hp, wp

    # ------------------------------------------------------------------ proj (roma_models.py:156-169)
    def proj_from_padded(self, s, tap, E, h, w, tag):
        """1x1 conv + folded BN on a zero-padded tap -> compact channels-last [E, h, w, cout]."""
        cin, cout = arch.PROJ[s]
        P = self.w.proj[s]
        out = self.buf(f"proj{tag}.{s}", (E, h, w, pad8(cout)), zero=True)
        rows = E * (h + 2) * (w + 2)
        self.gemm(tap, P["w"], out, rows, cout, cin, cin, P["w"].shape[1], pad8(cout), bias=P["b"],
                  rowmap=cabi.ROWMAP_PAD_TO_COMPACT, pad_h=h + 2, pad_w=w + 2)
        return out

    # ------------------------------------------------------------------ GP + transformer decoder (scale 16)
    def coarse_match(self, feat16, E, D, b, hp, wp, state):
        """GP posterior (matcher.py:291-323), embedding decoder (transformer/__init__.py:30-46) and
        cls_to_flow_refine (utils.py:300-322): fills state [D, hp, wp, 3]; returns the projected features."""
        n = hp * wp
        cin, cf = arch.PROJ[16]
        P = self.w.proj[16]
        f32 = cabi.RB_F32
        p16 = self.buf("gp.p16", (E * n, cf), dtype=torch.float32)      # GP runs in fp32 (x.float(), matcher.py:296)
        with self.stage("  gp.proj16"):
            self.gemm(feat16, P["w"], p16, E * n, cf, cin, cin, P["w"].shape[1], cf, dtype_c=f32, bias=P["b"])
        norms = self.buf("gp.norms", (E * n,), dtype=torch.float32)
        call("romab200_row_norms", "rb_rownorm_args", x=p16, out=norms, rows=E * n, cols=cf, ldx=cf, dtype=f32)
        ldw = pad8(n)
        nrhs = arch.GP_DIM
        Wk = self.buf("gp.work", (E, n + nrhs, ldw), dtype=torch.float32)
        stride_w = (n + nrhs) * ldw
        # K_yy + sigma*I for every image (its own features): exp((cos-1)/T)   (matcher.py:191-200, 298, 301)
        gp_split = self.split or (self.dtype != torch.float32 and self.gp_tensor_core)     # GP contractions as split-fp16 pairs (fp32-class)
        tc_kernel = False                 # (the K' = 3K operand trick of round 1 is superseded by the split back-end)
        xs = None
        if gp_split:
            # all-pairs CosKernel on tcgen05 with fp32-class accuracy: the L2-normalised rows as an RB_F16S pair
            with self.stage("  gp.split"):
                xs = self.split_pair(p16, E * n, cf, cf, name="gp.xs", row_norm=norms)
        elif tc_kernel:
            # all-pairs CosKernel on the f16 tensor pipe with fp32-class accuracy: L2-normalised rows split into fp16
            # hi/lo parts, A' = [hi|lo|hi], B' = [hi|hi|lo]  ->  A'.B'^T = hi.hi + lo.hi + hi.lo  (K' = 3*512)
            xa = self.buf("gp.split_a", (E * n, 3 * cf), dtype=torch.float16)
            xb = self.buf("gp.split_b", (E * n, 3 * cf), dtype=torch.float16)
            with self.stage("  gp.split"):
                call("romab200_split_f16x3", "rb_split_args", x=p16, dst=xa, rows=E * n, cols=cf, ldx=cf, ldd=3 * cf, row_norm=norms, layout_b=0)
                call("romab200_split_f16x3", "rb_split_args", x=p16, dst=xb, rows=E * n, cols=cf, ldx=cf, ldd=3 * cf, row_norm=norms, layout_b=1)
        self._corr16 = None
        if self.split and self.lc_table16:
            # the stride-16 refiner's local correlation (r = 7: 256 dot products of 512 channels per pixel) from ONE all-pairs
            # contraction per direction on tcgen05: table[i, p, q] = <x_i[p], y_i[q]> / sqrt(512), gathered by the prologue
            with self.stage("  gp.corr16"):
                ps = self.split_pair(p16, E * n, cf, cf, name="gp.p16s")
                tab = self.buf("ref.corr16", (D, n, ldw), dtype=torch.float32)
                for i0, cnt, y0 in ([(0, b, b)] if D == b else [(0, b, b), (b, b, 0)]):
                    self.gemm(ps.at(i0 * n * cf), ps.at(y0 * n * cf), tab.data_ptr() + i0 * n * ldw * 4, n, n, cf, cf, cf, ldw, dtype_c=f32,
                              batch0=cnt, sa0=n * cf, sb0=n * cf, sc0=n * ldw, alpha=float(torch.rsqrt(torch.tensor(float(cf)))))
                self._corr16 = (tab, ldw)
        with self.stage("  gp.kyy"):
            if gp_split:
                self.gp_kernel_matrix_split(xs, xs, norms, norms, Wk, n, cf, ldw, batch=E, sa=n * cf, sb=n * cf, sc=stride_w,
                                            sna=n, snb=n, diag=arch.GP_SIGMA_NOISE)
            elif tc_kernel:
                self.gp_kernel_matrix_tc(xa, xb, norms, norms, Wk, n, cf, ldw, batch=E, sa=n * 3 * cf, sb=n * 3 * cf, sc=stride_w,
                                         sna=n, snb=n, diag=arch.GP_SIGMA_NOISE)
            else:
                self.gp_kernel_matrix(p16, p16, norms, norms, Wk, n, cf, ldw, batch=E, sa=n * cf, sb=n * cf, sc=stride_w,
                                      sna=n, snb=n, diag=arch.GP_SIGMA_NOISE)
        basis_t = self.gp_basis_t(hp, wp)
        for e in range(E):
            self.copy2d(basis_t, Wk.data_ptr() + (e * stride_w + n * ldw) * 4, nrhs, n, n, ldw, f32, f32)
        with self.stage("  gp.solve"):
            # algo 2: 128-wide blocks factored in shared memory + explicit block inverses, everything else K=128 GEMMs
            ws_bytes = max((E * ((n + 31) // 32) * 1024 + 1) * 4, E * ((n + 127) // 128) * 65536)
            if self.gp_algo == 3:
                ws_bytes = E * (((n + 127) // 128) * 65536 + 4 * max((n + nrhs) * 128 + 16384, nrhs * 128 + 16384 + 128 * ldw))
            ws = self.buf("gp.solve_ws", (ws_bytes // 4,), dtype=torch.float32)
            call("romab200_gp_solve", "rb_gp_solve_args", W=Wk, n=n, nrhs=nrhs, batch=E, ldw=ldw, stride=stride_w,
                 workspace=ws if self.gp_algo else None, workspace_bytes=ws_bytes if self.gp_algo else 0, algo=self.gp_algo)
        # K_xy and mu = K_xy @ alpha for every decoder item: query image i, support image (i + b) % E
        dim = arch.DEC_DIM
        tokens = self.buf("dec.tokens_in", (D * n, dim))
        es = tokens.element_size()
        halves = [(0, b, b)] if D == b else [(0, b, b), (b, b, 0)]     # (first item, count, first support image)
        if gp_split:
            kxy = self.sbuf("gp.kxy", (D, n, ldw))
            alpha = self.sbuf("gp.alpha", (E, nrhs, ldw))
            with self.stage("  gp.kxy+mu"):
                for e in range(E):          # alpha^T = rows n.. of every solved workspace
                    call("romab200_split_f16s", "rb_split_pair_args", x=Wk.data_ptr() + (e * stride_w + n * ldw) * 4,
                         hi=alpha.at(e * nrhs * ldw).hi, lo=alpha.at(e * nrhs * ldw).lo, rows=nrhs, cols=n, ldx=ldw, ldd=ldw)
                for i0, cnt, y0 in halves:
                    self.gp_kernel_matrix_split(xs.at(i0 * n * cf), xs.at(y0 * n * cf), norms.data_ptr() + i0 * n * 4, norms.data_ptr() + y0 * n * 4,
                                                kxy.at(i0 * n * ldw), n, cf, ldw, batch=cnt, sa=n * cf, sb=n * cf, sc=n * ldw, sna=n, snb=n, diag=0.0)
                    self.gemm(kxy.at(i0 * n * ldw), alpha.at(y0 * nrhs * ldw), tokens.data_ptr() + i0 * n * dim * es, n, nrhs, n, ldw, ldw, dim,
                              batch0=cnt, sa0=n * ldw, sb0=nrhs * ldw, sc0=n * dim)
            halves = []
        else:
            kxy = self.buf("gp.kxy", (D, n, ldw), dtype=torch.float32)
        for i0, cnt, y0 in halves:
          with self.stage("  gp.kxy+mu"):
            if tc_kernel:
                self.gp_kernel_matrix_tc(xa.data_ptr() + i0 * n * 3 * cf * 2, xb.data_ptr() + y0 * n * 3 * cf * 2,
                                         norms.data_ptr() + i0 * n * 4, norms.data_ptr() + y0 * n * 4,
                                         kxy.data_ptr() + i0 * n * ldw * 4, n, cf, ldw, batch=cnt, sa=n * 3 * cf, sb=n * 3 * cf,
                                         sc=n * ldw, sna=n, snb=n, diag=0.0)
            else:
                self.gp_kernel_matrix(p16.data_ptr() + i0 * n * cf * 4, p16.data_ptr() + y0 * n * cf * 4,
                                      norms.data_ptr() + i0 * n * 4, norms.data_ptr() + y0 * n * 4,
                                      kxy.data_ptr() + i0 * n * ldw * 4, n, cf, ldw, batch=cnt, sa=n * cf, sb=n * cf, sc=n * ldw,
                                      sna=n, snb=n, diag=0.0)
            self.gemm(kxy.data_ptr() + i0 * n * ldw * 4, Wk.data_ptr() + (y0 * stride_w + n * ldw) * 4,
                      tokens.data_ptr() + i0 * n * dim * es, n, nrhs, n, ldw, ldw, dim, dtype_ab=f32,
                      batch0=cnt, sa0=n * ldw, sb0=stride_w, sc0=n * dim)
        # tokens = cat(gp_posterior, f1_s) (transformer/__init__.py:33)
        self.copy2d(p16, tokens.data_ptr() + arch.GP_DIM * es, D * n, cf, cf, dim, f32, self.dt)
        if self.debug is not None:
            self.debug["gp.mu"] = tokens.view(D, n, dim)[:, :, :arch.GP_DIM].float().clone()
        x = self.buf("dec.x", (D * n, dim), dtype=torch.float32)
        self.copy2d(tokens, x, D * n, dim, dim, dim, self.dt, f32)
        with self.stage("  dec.blocks"):
            for blk in self.w.dec:
                self.block(x, blk, D, n, dim, arch.DEC_HEADS, arch.DEC_MLP, arch.DEC_LN_EPS, "dec")
        if self.split:
            xa = x                                  # split into an RB_F16S pair by the GEMM wrapper
        else:
            xa = self.buf("dec.xa", (D * n, dim))
            self.copy2d(x, xa, D * n, dim, dim, dim, f32, self.dt)
        ldl = pad8(arch.CLS_OUT)
        logits = self.buf("dec.logits", (D * n, ldl), dtype=torch.float32)
        with self.stage("  dec.to_out+cls"):
            self.gemm(xa, self.w.to_out_w, logits, D * n, arch.CLS_OUT, dim, dim, dim, ldl, dtype_c=f32, bias=self.w.to_out_b)
            call("romab200_cls_to_flow_refine", "rb_cls_args", logits=logits, state=state, rows=D * n, ldl=ldl,
                 res=arch.CLS_RES, dtype=f32)
        if self.debug is not None:
            self.debug["cls"] = logits.view(D, n, ldl)[:, :, :arch.CLS_OUT].clone()
        # the stride-16 refiner consumes the same projected features (matcher.py:450,484-486)
        feat = self.buf("proj.16", (E, hp, wp, cf))
        self.copy2d(p16, feat, E * n, cf, cf, cf, f32, self.dt)
        return feat

    def gp_kernel_matrix(self, A, B, na, nb, C, n, cf, ldc, batch, sa, sb, sc, sna, snb, diag):
        """C[z] = exp((cos(A[z], B[z]) - 1) / T) + diag*I  — the all-pairs CosKernel contraction."""
        self.gemm(A, B, C, n, n, cf, cf, cf, ldc, dtype_ab=cabi.RB_F32, dtype_c=cabi.RB_F32, batch0=batch,
                  sa0=sa, sb0=sb, sc0=sc, epi=cabi.EPI_COSKERNEL, norm_a=na, norm_b=nb, sna0=sna, snb0=snb,
                  eps=arch.GP_COS_EPS, inv_t=1.0 / arch.GP_TEMPERATURE, diag_add=diag, cos_normalized=0)

    def gp_kernel_matrix_split(self, A: Split, B: Split, na, nb, C, n, cf, ldc, batch, sa, sb, sc, sna, snb, diag):
        """Same contraction on tcgen05 from RB_F16S pairs of the L2-normalised rows (cos_normalized=1); C fp32 or a pair."""
        self.gemm(A, B, C, n, n, cf, cf, cf, ldc, dtype_c=cabi.RB_F32, batch0=batch,
                  sa0=sa, sb0=sb, sc0=sc, epi=cabi.EPI_COSKERNEL, norm_a=na, norm_b=nb, sna0=sna, snb0=snb,
                  eps=arch.GP_COS_EPS, inv_t=1.0 / arch.GP_TEMPERATURE, diag_add=diag, cos_normalized=1)

    def gp_kernel_matrix_tc(self, A, B, na, nb, C, n, cf, ldc, batch, sa, sb, sc, sna, snb, diag):
        """Same contraction on tcgen05 from the split fp16 operands (pre-normalised rows: cos_normalized=1)."""
        self.gemm(A, B, C, n, n, 3 * cf, 3 * cf, 3 * cf, ldc, dtype_ab=cabi.RB_F16, dtype_c=cabi.RB_F32, batch0=batch,
                  sa0=sa, sb0=sb, sc0=sc, epi=cabi.EPI_COSKERNEL, norm_a=na, norm_b=nb, sna0=sna, snb0=snb,
                  eps=arch.GP_COS_EPS, inv_t=1.0 / arch.GP_TEMPERATURE, diag_add=diag, cos_normalized=1)

    # ------------------------------------------------------------------ ConvRefiner (matcher.py:124-179)
    def refine(self, s, feat, ldf, E, D, b, h, w, state, scale_factor, h1, w1, tag):
        R = self.w.refiner[s]
        spec, c, cp = R["spec"], R["c"], R["cp"]
        d = self.buf(f"ref.d.{tag}", (D * h * w, cp), zero=True)
        t = None if self.split else self.buf(f"ref.t.{tag}", (D * h * w, cp), zero=True)
        r = spec.radius
        tiles = None
        table, ld_table = (self._corr16 if s == 16 and getattr(self, "_corr16", None) else (None, 0))
        if r in self.lc_tile_radii and self.dt == cabi.RB_F32 and table is None:
            # workspace of the tile-cooperative pass (coherent flow: one CTA per 8x2 / 8x4 pixels stages the union of their windows)
            tiles = self.buf(f"ref.tiles.{tag}", (D * cabi.prologue_tiles(r, h, w),), dtype=torch.uint8, zero=True)
        with self.stage(f"  prologue{s}.{tag[:2]}"):
          call("romab200_refiner_prologue", "rb_refiner_prologue_args", feat=feat, ldf=ldf, n_img=E, y_shift=b,
             tile_done=tiles, tile_done_len=tiles.numel() if tiles is not None else 0, corr_table=table, ld_corr_table=ld_table,
             state=state, d=d, ldd=cp, D=D, h=h, w=w, cf=spec.feat, emb=spec.emb, radius=r, dtype=self.dt,
             emb_weight=R["emb_w"], emb_bias=R["emb_b"],
             disp_scale=float(torch.tensor(40 / 32 * scale_factor, dtype=torch.float32)),
             grid_x=self.grid_axis(w), grid_y=self.grid_axis(h),
             win_x=self.window_axis(r, w) if r else None, win_y=self.window_axis(r, h) if r else None)
        if self.debug is not None:
            self.debug[f"{tag}.refiner_in"] = d.view(D, h, w, cp)[..., :c].float().clone()
        rows = D * h * w
        if c == 24 and (self.dtype != torch.float32 or self.fused_small_f32):
            # thin stride-1 maps: one fused DW5x5+ReLU+PW kernel per block, ping-ponging between the two buffers
            # (fp32 maps: fp32 FFMA throughout, the arithmetic of the un-fused fp32 path)
            if t is None:
                t = self.buf(f"ref.t.{tag}", (D * h * w, cp), zero=True)
            for blk in R["blocks"]:
                call("romab200_refiner_block_small", "rb_refiner_block_small_args", **{"in": d}, out=t, ld=cp, dw_weight=blk["dw_w"],
                     ldw=cp, dw_bias=blk["dw_b"], pw_weight_host=blk["pw_w_host"].data_ptr(), pw_bias_host=blk["pw_b_host"].data_ptr(), batch=D, h=h, w=w, c=c, dtype=self.dt)
                d, t = t, d
        elif c == 144 and self.dtype != torch.float32 and self.fused_c144:
            # stride-2 maps: depthwise stage on the CUDA cores feeding a tcgen05 pointwise GEMM inside one kernel
            for blk in R["blocks"]:
                call("romab200_refiner_block_c144", "rb_refiner_block_c144_args", **{"in": d}, out=t, ld=cp, dw_weight=blk["dw_w"], ldw=cp,
                     dw_bias=blk["dw_b"], pw_weight=blk["pw_w"], ld_pw=cp, pw_bias=blk["pw_b"], batch=D, h=h, w=w, c=c, dtype=self.dt)
                d, t = t, d
        elif c == 144 and self.split and self.fused_c144_f32:
            # parity mode, stride-2 maps: the same fused block on fp32 maps with the split-fp16 pointwise GEMM (bit-identical
            # to the depthwise kernel + split GEMM pair below, at one read and one write of the map instead of four transfers)
            if t is None:
                t = self.buf(f"ref.t.{tag}", (D * h * w, cp), zero=True)
            for blk in R["blocks"]:
                call("romab200_refiner_block_c144", "rb_refiner_block_c144_args", **{"in": d}, out=t, ld=cp, dw_weight=blk["dw_w"], ldw=cp,
                     dw_bias=blk["dw_b"], pw_weight=blk["pw_w"].hi, pw_weight_lo=blk["pw_w"].lo, ld_pw=cp, pw_bias=blk["pw_b"],
                     batch=D, h=h, w=w, c=c, dtype=cabi.RB_F32)
                d, t = t, d
        elif self.split:
            # parity mode: fp32 maps; the depthwise kernel writes its result as the RB_F16S A operand of the pointwise GEMM
            ts = self.sbuf(f"ref.ts.{tag}", (D * h * w, cp), zero=True)
            for blk in R["blocks"]:
                call("romab200_dwconv5x5_relu", "rb_dwconv_args", **{"in": d}, out=ts.hi, out_lo=ts.lo, ldi=cp, ldo=cp, weight=blk["dw_w"], ldw=cp,
                     bias=blk["dw_b"], batch=D, h=h, w=w, c=c, dtype=cabi.RB_F32)
                self.gemm(ts, blk["pw_w"], d, rows, c, c, cp, cp, cp, bias=blk["pw_b"])
        else:
            for blk in R["blocks"]:
                call("romab200_dwconv5x5_relu", "rb_dwconv_args", **{"in": d}, out=t, ldi=cp, ldo=cp, weight=blk["dw_w"], ldw=cp,
                     bias=blk["dw_b"], batch=D, h=h, w=w, c=c, dtype=self.dt)
                self.gemm(t, blk["pw_w"], d, rows, c, c, cp, cp, cp, bias=blk["pw_b"])
        delta = self.buf(f"ref.delta.{tag}", (rows, 3), dtype=torch.float32) if self.debug is not None else None
        call("romab200_refiner_tail", "rb_refiner_tail_args", d=d, ldd=cp, weight=R["out_w"], ldw=cp, bias=R["out_b"],
             state=state, rows=rows, c=c, scale_x=s / (arch.REFINE_INIT * w1), scale_y=s / (arch.REFINE_INIT * h1),
             dtype=self.dt, delta_out=delta)
        if self.debug is not None:
            self.debug[f"{tag}.delta"] = delta.view(D, h, w, 3).clone()

    def resize_state(self, src, D, hi, wi, ho, wo, name):
        dst = self.buf(name, (D, ho, wo, 3), dtype=torch.float32)
        call("romab200_bilinear_resize", "rb_resize_args", **{"in": src}, out=dst, batch=D, hi=hi, wi=wi, ho=ho, wo=wo, c=3)
        return dst

    # ------------------------------------------------------------------ one pass of the matcher
    def encode_cnn(self, images: torch.Tensor, tag: str):
        """VGG19 pyramid + proj[s] of one pass: {s: (projected channels-last features, pitch)}, {s: (h, w)}."""
        E = images.shape[0]
        with self.stage(f"vgg.{tag}"):
            taps = self.vgg(images, tag)
        sizes = {s: (taps[s][1], taps[s][2]) for s in (1, 2, 4, 8)}
        feats = {}
        for s in (8, 4, 2, 1):
            h, w = sizes[s]
            with self.stage(f"proj{s}.{tag}"):
                feats[s] = (self.proj_from_padded(s, taps[s][0], E, h, w, tag), pad8(arch.PROJ[s][1]))
        return feats, sizes

    def run_pass(self, images: torch.Tensor, b: int, symmetric: bool, upsample: bool, scale_factor: float,
                 state_in: Optional[Tuple[torch.Tensor, int, int]] = None, keep_states=False, cnn=None, cnn_ready=None, vit=None):
        """images [2b,3,H,W] fp32 (A batch then B batch).  Returns (state [D,H,W,3], states per scale, sizes).
        `cnn` = result of `encode_cnn` computed elsewhere (side stream); `cnn_ready` = event to wait for before use."""
        tag = "up" if upsample else "lo"
        E = 2 * b
        D = E if symmetric else b
        _, _, H, W = images.shape
        if cnn is None and (upsample or vit is None):
            cnn = self.encode_cnn(images, tag)
        if not upsample and vit is None:
            with self.stage("dinov2"):
                vit = self.dinov2(images)
        if cnn is None:
            cnn = self.encode_cnn(images, tag)
        feats, sizes = cnn
        sizes = dict(sizes)
        states = {}
        if not upsample:
            feat16_raw, hp, wp = vit
            sizes[16] = (hp, wp)
            state = self.buf("state.lo.16", (D, hp, wp, 3), dtype=torch.float32)
            with self.stage("gp+decoder"):
                feat16 = self.coarse_match(feat16_raw, E, D, b, hp, wp, state)
            if self.debug is not None:
                self.debug["coarse_state"] = state.clone()
            scales = arch.SCALES
        else:
            src, hi, wi = state_in
            state = self.resize_state(src, D, hi, wi, *sizes[8], name="state.up.8")
            scales = arch.UPSAMPLE_SCALES
        for s in scales:
            h, w = sizes[s]
            if s == 16:
                feat, ldf = feat16, arch.PROJ[16][1]
            else:
                if cnn_ready is not None:
                    torch.cuda.current_stream().wait_event(cnn_ready)
                    cnn_ready = None
                feat, ldf = feats[s]
            if self.debug is not None:
                self.debug[f"{tag}.proj{s}"] = feat.view(E, h, w, -1)[..., :arch.PROJ[s][1]].float().clone()
            with self.stage(f"refine{s}.{tag}"):
                self.refine(s, feat, ldf, E, D, b, h, w, state, scale_factor, H, W, f"{tag}{s}")
            if keep_states or s == 16:
                states[s] = state.clone() if keep_states else state
            if s != 1:
                ho, wo = sizes[s // 2]
                state = self.resize_state(state, D, h, w, ho, wo, name=f"state.{tag}.{s // 2}")
        return state, states, sizes

    def run_match(self, images, images_hi, b, symmetric, scale_lo, scale_hi, attenuate, warp, cert):
        """Device side of match(): coarse pass, optional upsample pass, epilogue — no allocation, no host sync.
        The CNN branch (VGG19 + proj of both passes) has no dependency on the ViT / GP / decoder chain, so it runs on a
        side stream and overlaps the latency-bound GP solve and decoder; under CUDA-graph capture this becomes a fork."""
        main = torch.cuda.current_stream()
        if self._side is None:
            self._side = torch.cuda.Stream(device=self.device)
        side = self._side
        overlap = self.overlap_cnn and self.debug is None
        cnn_lo = cnn_hi = ev_lo = ev_hi = vit = None
        if overlap:
            # the ViT saturates the tensor pipe by itself; the CNN branch is released when it finishes, so that it
            # fills the SMs left idle by the latency-bound GP solve and the small decoder GEMMs that follow
            with self.stage("dinov2"):
                vit = self.dinov2(images)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                self._lane = "side"
                cnn_lo = self.encode_cnn(images, "lo")
                ev_lo = torch.cuda.Event()
                ev_lo.record(side)
                if images_hi is not None:
                    cnn_hi = self.encode_cnn(images_hi, "up")
                    ev_hi = torch.cuda.Event()
                    ev_hi.record(side)
                self._lane = "main"
        hs, ws = images.shape[-2:]
        state, states, sizes = self.run_pass(images, b, symmetric, False, scale_lo, cnn=cnn_lo, cnn_ready=ev_lo, vit=vit)
        coarse = states[16] if attenuate else None
        hc, wc = sizes[16]
        if images_hi is not None:
            hh, wh = images_hi.shape[-2:]
            state, _, _ = self.run_pass(images_hi, b, symmetric, True, scale_hi, (state, hs, ws), cnn=cnn_hi, cnn_ready=ev_hi)
            hs, ws = hh, wh
        self.epilogue(state, coarse, hc, wc, b, hs, ws, symmetric, out=(warp, cert))

    def epilogue(self, state, coarse_state, hc, wc, b, H, W, symmetric, out=None):
        Wout = 2 * W if symmetric else W
        if out is None:
            warp = torch.empty(b, H, Wout, 4, dtype=torch.float32, device=self.device)
            cert = torch.empty(b, H, Wout, dtype=torch.float32, device=self.device)
        else:
            warp, cert = out
            assert warp.shape == (b, H, Wout, 4) and cert.shape == (b, H, Wout)
        call("romab200_match_epilogue", "rb_match_epilogue_args", state=state, coarse_state=coarse_state, hc=hc, wc=wc,
             warp=warp, cert=cert, b=b, H=H, W=W, symmetric=int(symmetric), grid_x=self.grid_axis(W), grid_y=self.grid_axis(H))
        return warp, cert

    def kde(self, x: torch.Tensor, std: float = 0.1, half: bool = True):
        x = x.contiguous().float()
        n = x.shape[0]
        out = torch.empty(n, dtype=torch.float32, device=x.device)
        splits = 16 if n >= 8192 else 1
        sym = bool(half) and splits > 1 and self.kde_symmetric      # every pair once: (splits + blocks of 256) * n floats of workspace
        nws = (splits + (n + 255) // 256) * n if sym else splits * n
        ws = torch.empty(nws, dtype=torch.float32, device=x.device) if splits > 1 else None
        call("romab200_kde_density", "rb_kde_args", x=x, density=out, n=n, std=std, half=int(half), workspace=ws, splits=splits,
             symmetric=int(sym), workspace_floats=nws if ws is not None else 0)
        return out
