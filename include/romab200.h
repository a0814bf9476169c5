/*
 * romab200.h — C ABI of the B200-native RoMa dense-matching kernels (libromab200.so).
 *
 * Drop-in boundary for ONE path: RoMa's dense match()/sample() inference.  The reference
 * (Parskatt/RoMa) is pure Python/PyTorch; the only native operator boundary it has on this path is
 * the optional third-party wheel `local_corr.local_corr` (romatch/utils/local_correlation.py:22-35).
 * Every entry point below cites the reference code it replaces.  Conventions:
 *
 *   - plain pointers and sizes only (no torch types); every pointer is DEVICE memory owned by the
 *     caller (PyTorch's allocator in the host package); nothing is allocated or synchronised inside;
 *   - every call enqueues work on the given CUDA stream (a `cudaStream_t` passed as void*) and returns
 *     immediately: 0 = ok, non-zero = error, message via romab200_last_error() (thread-local);
 *   - activations are channels-last ("NHWC"): a [B,H,W,C] map is a row-major [B*H*W, C] matrix with an
 *     explicit row pitch, so 1x1 convolutions and Linear layers are the same GEMM;
 *   - dtypes: RB_F32 / RB_F16 / RB_BF16; accumulation is always fp32.
 *   - RB_F16S ("split fp16 pair") is the storage format of the tensor-core parity mode: a matrix is held as TWO fp16
 *     planes of the same pitch, hi = fp16(x) and lo = fp16((x - hi) * 2^11), value = hi + lo * 2^-11: 22 significand bits
 *     with the exponent range of fp16 (the reference's own CUDA autocast range).  romab200_gemm contracts such operands
 *     with three tcgen05 MMAs per k-step (hi.hi + 2^-11 (hi.lo + lo.hi), fp32 accumulation in TMEM), which reproduces an
 *     fp32 GEMM to ~2^-22 relative; arguments named *_lo carry the second plane.
 */
#ifndef ROMAB200_H
#define ROMAB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ROMAB200_ABI_VERSION 4

enum rb_dtype { RB_F32 = 0, RB_F16 = 1, RB_BF16 = 2, RB_F16S = 3 };
enum rb_act { RB_ACT_NONE = 0, RB_ACT_RELU = 1, RB_ACT_GELU = 2 };
enum rb_rowmap { RB_ROWMAP_NONE = 0, RB_ROWMAP_PAD_KEEP = 1, RB_ROWMAP_PAD_TO_COMPACT = 2, RB_ROWMAP_SEGMENT = 3 };
enum rb_epi { RB_EPI_LINEAR = 0, RB_EPI_COSKERNEL = 1 };
enum rb_backend { RB_BACKEND_AUTO = 0, RB_BACKEND_SIMT = 1, RB_BACKEND_TCGEN05 = 2 };

int romab200_abi_version(void);
const char* romab200_last_error(void);
/* number of CUDA kernels this library has launched so far in this process */
unsigned long long romab200_launch_count(void);
/* 1 if the running device is sm_100 (B200) and the tcgen05/TMA kernels may be launched */
int romab200_device_ok(void);

/* ------------------------------------------------------------------------------------------------
 * GEMM with fused epilogue:  C[m,n] = epi( sum_k A[m + tap(k), k] * B[n,k] )
 *
 * Replaces every nn.Linear / 1x1 nn.Conv2d (+ folded BatchNorm) / 3x3 nn.Conv2d on the path:
 *   ViT + decoder Linear layers      romatch/models/transformer/layers/{attention.py:50-63,mlp.py:35-41}
 *   proj[s] 1x1 conv + BN            romatch/models/model_zoo/roma_models.py:156-169 (matcher.py:441-450)
 *   ConvRefiner pointwise convs      romatch/models/matcher.py:121 (create_block conv2)
 *   VGG19-BN 3x3 conv + BN + ReLU    romatch/models/encoders.py:17-27 (as a 9-tap shifted GEMM on a
 *                                    zero-padded NHWC map: tap t reads rows m + tap_rows[t])
 *   CosKernel all-pairs contraction  romatch/models/matcher.py:191-200 (RB_EPI_COSKERNEL)
 *   attention QK^T / PV, GP K_xy@alpha, Cholesky trailing updates (batched, strided)
 *
 * A: [M, K] row-major (pitch lda).  B: [N, K] row-major (pitch ldb), or [K, N] when trans_b != 0.
 * K = ntaps * k_per_tap; element k belongs to tap k / k_per_tap and reads A row m + tap_rows[tap]
 * (rows outside [0, a_rows) read as zero).  Batching: grid over batch0 x batch1 with element strides.
 *
 * Epilogue RB_EPI_LINEAR:    v = alpha*acc + bias[n]; v = act(v); v *= col_scale[n]; v += R[m,n]
 * Epilogue RB_EPI_COSKERNEL: c = acc * s(m,n), s = 1/(na[m]*nb[n]+eps)            (cos_normalized == 0)
 *                                              s = na[m]*nb[n]/(na[m]*nb[n]+eps)  (operands pre-normalised)
 *                            v = exp((c - 1) * inv_t) + (m == n ? diag_add : 0)
 * Row map of the store: NONE; PAD_KEEP (m indexes a zero-padded [*,pad_h,pad_w] grid; border rows are not
 * computed: they are left alone or rewritten with zeros, the value they hold in every map of the path); PAD_TO_COMPACT (same, interior rows are written to the un-padded row index);
 * SEGMENT (row m -> (m / seg_in) * seg_out + m % seg_in + seg_off).
 * Output pitch: the tcgen05 back-end stores tiles with TMA when ldc (and the batch strides) are multiples of 16 bytes; TMA clips at
 * 16-byte granules, so the pad columns N .. roundup(N, 16 bytes) of a written row receive zeros (columns beyond are untouched).
 * ------------------------------------------------------------------------------------------------ */
typedef struct {
    const void* A; const void* B; void* C;
    int32_t M, N, K;
    int64_t lda, ldb, ldc;
    int32_t dtype_ab, dtype_c;
    int32_t trans_b;
    int32_t batch0, batch1;
    int64_t sa0, sa1, sb0, sb1, sc0, sc1;
    int32_t ntaps; int32_t tap_rows[9]; int64_t a_rows;
    float alpha;
    const float* bias; const float* col_scale;
    const void* R; int64_t ldr, sr0, sr1; int32_t dtype_r;
    int32_t act;
    int32_t epi;
    const float* norm_a; const float* norm_b; int64_t sna0, snb0;
    float eps, inv_t, diag_add; int32_t cos_normalized;
    int32_t rowmap, pad_h, pad_w, seg_in, seg_out, seg_off;
    int32_t backend;
    /* second planes of RB_F16S operands / output (dtype_ab == RB_F16S: A_lo and B_lo, same geometry as A and B;
       dtype_c == RB_F16S: C_lo, same pitch as C); NULL otherwise */
    const void* A_lo; const void* B_lo; void* C_lo;
    /* tcgen05 back-end: upper bound on the persistent grid (0 = one CTA per SM).  A GEMM running on a side stream beside a chain of short
       dependent kernels (the GP solve) leaves the remaining SMs free, so that those kernels start without waiting for a whole GEMM. */
    int32_t max_ctas;
} rb_gemm_args;
int romab200_gemm(const rb_gemm_args* args, void* stream);

/* LayerNorm over the last dim (nn.LayerNorm in block.py:50 / dinov2.py:88): y = (x-mu)/sqrt(var+eps)*g + b */
typedef struct {
    const void* x; void* y; const float* gamma; const float* beta;
    int64_t rows; int32_t cols; int64_t ldx, ldy; int32_t dtype_x, dtype_y; float eps;
    void* y_lo;   /* second plane when dtype_y == RB_F16S */
} rb_layernorm_args;
int romab200_layernorm(const rb_layernorm_args* args, void* stream);

/* Row softmax of attention scores: s = softmax(scale * s) over `cols` (SDPA, attention.py:59); in place, or (out_hi != NULL,
 * dtype RB_F32) written as an RB_F16S pair of planes [rows, ldo] for the split-fp16 PV product (pad columns receive 0) */
typedef struct { void* s; int64_t rows; int32_t cols; int64_t lds; int32_t dtype; float scale;
                 void* out_hi; void* out_lo; int64_t ldo; } rb_softmax_args;
int romab200_softmax_rows(const rb_softmax_args* args, void* stream);

/* Fused attention forward (F.scaled_dot_product_attention, attention.py:50-63), 16-bit tensor-core path:
 * qkv [batch, n_tokens, ld_qkv] holds q | k | v (each heads*head_dim wide, heads contiguous); out [batch, n_tokens, ld_out].
 * out[b, i, h*d:(h+1)*d] = softmax_j(q_i . k_j / sqrt(d)) v_j.  head_dim 64 or 128. */
typedef struct {
    const void* qkv; void* out; int64_t ld_qkv, ld_out; int32_t batch, n_tokens, heads, head_dim, dtype;
    /* dtype == RB_F16S (head_dim 64): qkv and out are split-fp16 pairs, these are their second planes; fp32-class result */
    const void* qkv_lo; void* out_lo;
} rb_flash_attn_args;
int romab200_flash_attn(const rb_flash_attn_args* args, void* stream);

/* L2 norm of every row: out[r] = ||x[r,:]||  (CosKernel, matcher.py:192-194) */
typedef struct { const void* x; float* out; int64_t rows; int32_t cols; int64_t ldx; int32_t dtype; } rb_rownorm_args;
int romab200_row_norms(const rb_rownorm_args* args, void* stream);

/* Strided 2-D copy / cast: dst[r, c] = (dst_dtype) src[r, c] * scale[r]  (scale may be NULL) */
typedef struct {
    const void* src; void* dst; int64_t rows; int32_t cols; int64_t lds, ldd; int32_t dtype_src, dtype_dst;
    const float* row_scale; int32_t row_scale_reciprocal;
} rb_copy2d_args;
int romab200_copy2d(const rb_copy2d_args* args, void* stream);

/* fp16 hi/lo operand split for fp32-class accuracy on the f16 tensor pipe:
 * dst[r, 0:C] = hi, dst[r, C:2C] = lo (or hi), dst[r, 2C:3C] = hi (or lo) of x[r,:]/scale[r]
 * layout A: [hi | lo | hi], layout B: [hi | hi | lo]  so that A'.B'^T = hi.hi + lo.hi + hi.lo */
typedef struct {
    const float* x; void* dst; int64_t rows; int32_t cols; int64_t ldx, ldd; const float* row_norm;
    int32_t layout_b;
} rb_split_args;
int romab200_split_f16x3(const rb_split_args* args, void* stream);

/* fp32 matrix -> RB_F16S planes: hi[r,c] = fp16(v), lo[r,c] = fp16((v - hi) * 2^11), v = x[r,c] (/ row_norm[r] if given).
 * The producer of every split-fp16 GEMM operand that is not written in that format by its own kernel. */
typedef struct {
    const float* x; void* hi; void* lo; int64_t rows; int32_t cols; int64_t ldx, ldd; const float* row_norm;
} rb_split_pair_args;
int romab200_split_f16s(const rb_split_pair_args* args, void* stream);

/* ---- VGG19-BN pieces that are not GEMMs (encoders.py:17-27) ------------------------------------ */
/* First conv (3 -> 64) + folded BN + ReLU, NCHW fp32 image -> zero-padded NHWC [B,H+2,W+2,64] */
typedef struct {
    const float* image; void* out; const float* weight /* [64][27] folded */; const float* bias /* [64] */;
    int32_t batch, height, width, cout; int32_t dtype_out;
    void* out_lo;   /* second plane when dtype_out == RB_F16S */
} rb_conv_first_args;
int romab200_conv3x3_first(const rb_conv_first_args* args, void* stream);
/* 2x2/2 max-pool between zero-padded NHWC maps: [B,H+2,W+2,C] -> [B,H/2+2,W/2+2,C] */
typedef struct { const void* in; void* out; int32_t batch, height, width, channels, dtype;
                 const void* in_lo; void* out_lo; /* second planes when dtype == RB_F16S */ } rb_maxpool_args;
int romab200_maxpool2x2_padded(const rb_maxpool_args* args, void* stream);

/* ---- DINOv2 tokenisation (dinov2.py:192-201, patch_embed.py:69-82) ------------------------------ */
/* im2col of non-overlapping 14x14 patches: NCHW fp32 image -> [B*hp*wp, ldo] rows of (c,ky,kx) */
typedef struct { const float* image; void* out; int32_t batch, height, width, patch; int64_t ldo; int32_t dtype_out; } rb_im2col_args;
int romab200_im2col_patch(const rb_im2col_args* args, void* stream);
/* tokens[b,0,:] = cls + pos[0]; tokens[b,1+p,:] = patch[b,p,:] + pos[1+p]   (fp32 residual stream) */
typedef struct { const float* patch; const float* cls; const float* pos; float* tokens; int32_t batch, npatch, dim; } rb_tokens_args;
int romab200_assemble_tokens(const rb_tokens_args* args, void* stream);

/* ---- GP posterior (matcher.py:291-323): batched Cholesky + solves --------------------------------
 * W is a batch of workspaces [n + nrhs, n] (row-major, pitch ldw): rows 0..n-1 hold the SPD matrix
 * K_yy + sigma*I (lower triangle is read), rows n.. hold F^T ([nrhs, n]).  On return rows n.. hold
 * X^T where (K_yy + sigma I) X = F, i.e. alpha^T, ready to be the [N,K] operand of mu = K_xy @ alpha.
 * With algo 0 and 2 the lower triangle of rows 0..n-1 holds the Cholesky factor afterwards; the strict upper triangle is
 * unspecified (symmetric trailing updates only maintain the lower half).
 * Replaces torch.linalg.cholesky + torch.cholesky_solve (matcher.py:307-308). */
typedef struct {
    float* W; int32_t n, nrhs, batch; int64_t ldw, stride;
    void* workspace; int64_t workspace_bytes;
    int32_t algo;   /* 0: 32-wide panels, chain of small launches (no workspace)
                       1: the same as ONE cooperative persistent kernel; workspace >= (batch*ceil(n/32)*1024 + 1)*4 bytes
                       2: 128-wide blocks factored in shared memory with explicit block inverses, all O(n^2) work as K=128
                          GEMMs; workspace >= batch*ceil(n/128)*65536 bytes (receives the diagonal-block inverses)
                       3: the schedule of 2 with those GEMMs on the tensor cores (split-fp16 operand pairs, fp32-class; the symmetric
                          trailing update is an in-place TMA reduce-add); n % 4 == 0, ldw % 8 == 0, stride % 8 == 0; workspace >=
                          batch * (ceil(n/128)*65536 + 4*max((n+nrhs)*128 + 16384, nrhs*128 + 16384 + 128*ldw)) bytes */
} rb_gp_solve_args;
int romab200_gp_solve(const rb_gp_solve_args* args, void* stream);
/* ---- classifier head -> coarse flow (utils.py:300-322) ------------------------------------------
 * logits [rows, ldl] fp32/16 with 4096 anchor logits followed by the certainty logit; writes
 * state[row] = (flow_x, flow_y, certainty_logit). */
typedef struct { const void* logits; float* state; int64_t rows; int64_t ldl; int32_t res; int32_t dtype; } rb_cls_args;
int romab200_cls_to_flow_refine(const rb_cls_args* args, void* stream);

/* ---- ConvRefiner (matcher.py:124-179) ------------------------------------------------------------
 * feat: projected features of all encoder images [n_img, h, w, ldf] (channels-last, `cf` channels).
 * For decoder item i the query image is `i` and the support image is (i + y_shift) % n_img.
 * state: [D, h, w, 3] = (flow_x, flow_y, certainty_logit) fp32.
 * prologue writes d[D,h,w,ldd] = [x | grid_sample(y, flow) | disp_emb(40/32*sf*(flow-grid)) | local_corr | 0-pad]
 *   (matcher.py:132-168; local correlation per local_correlation.py:77-142 / local_corr.local_corr) */
typedef struct {
    const void* feat; int64_t ldf; int32_t n_img, y_shift;
    const float* state; void* d; int64_t ldd;
    int32_t D, h, w, cf, emb, radius; int32_t dtype;
    const float* emb_weight /* [emb][2] */; const float* emb_bias; float disp_scale;
    const float* grid_x; const float* grid_y;   /* linspace(-1+1/w, 1-1/w, w), linspace(-1+1/h, 1-1/h, h) (matcher.py:136-143) */
    const float* win_x; const float* win_y;     /* linspace(-2r/w, 2r/w, 2r+1), linspace(-2r/h, 2r/h, 2r+1) (local_correlation.py:93-103) */
    /* optional workspace (caller-owned, like every buffer): one byte per tile of the tile-cooperative pass for fp32 maps with a local
     * correlation (radius 7: 8x2 pixels (x by y), radius 3 / 2: 8x4 pixels per tile; D * ceil(h/Ty) * ceil(w/Tx) tiles).  When given, tiles whose
     * windows overlap (coherent flow) are produced by one CTA from a shared-memory copy of the union of their windows; the rest by the
     * per-pixel kernel.  NULL: per-pixel kernel only.  Same results either way up to the summation order of the dot products. */
    void* tile_done; int32_t tile_done_len;
    /* optional all-pairs table (radius > 0): corr_table[(item*h*w + p) * ld_corr_table + q] = <x[item, p, :], y[item, q, :]> / sqrt(cf) for every
     * position q of the other map, e.g. one romab200_gemm per direction at the coarsest scale, where the table is small (h*w = 1600) and the
     * contraction is the one the GP kernel matrix performs anyway (matcher.py:298-300).  The window dot products then are a gather of
     * (2r+2)^2 table entries per pixel instead of (2r+2)^2 * cf multiply-adds.  NULL: the dot products are computed here. */
    const float* corr_table; int64_t ld_corr_table;
} rb_refiner_prologue_args;
int romab200_refiner_prologue(const rb_refiner_prologue_args* args, void* stream);

/* Stand-alone local correlation with the reference wheel's semantics (local_correlation.py:22-35):
 * corr[b, p, k] = sum_c f0[b,p,c] * bilinear(f1[b], flow[b,p] + window[k])  (f0 already scaled by caller or
 * `scale` applied here), zero padding, k = (dy+r)*(2r+1) + (dx+r).  out pitch ldo (channels-last slice). */
typedef struct {
    const void* f0; const void* f1; int64_t ldf0, ldf1; int64_t f0_img_stride, f1_img_stride;
    const float* flow; int64_t ldflow; void* out; int64_t ldo;
    int32_t batch, h, w, c, radius; float scale; int32_t dtype_f, dtype_out;
    int32_t n_img, y_shift;   /* f1 image of item i = (i + y_shift) % n_img ; f0 image = i */
    const float* win_x; const float* win_y;   /* window offsets in normalised coordinates, 2r+1 each */
} rb_local_corr_args;
int romab200_local_corr(const rb_local_corr_args* args, void* stream);

/* The fused-local-corr wheel's operator, signature for signature (`local_corr.local_corr`, local_correlation.py:22-35):
 * out[b, p, k] = sum_c f0[b, p, c] * sample(f1[b], warp[b, p, k, :]), sample = bilinear (mode 0) or nearest (mode 1) lookup at the
 * normalised (x, y) position, align_corners=False, zero padding (grid_sample semantics); f0 is used as given (the caller pre-scales
 * by 1/sqrt(C) like `local_corr_wrapper` does).  f0 [B, HW, C] fp32 (pitch ldf0), f1 [B, H, W, C] fp32 channels-last (pitch ldf1),
 * warp [B, HW, K, 2] fp32 contiguous, out [B, HW, K] fp32 contiguous.  Arbitrary warps: nothing is assumed about a window lattice. */
typedef struct {
    const float* f0; const float* f1; int64_t ldf0, ldf1; const float* warp; float* out;
    int32_t batch, h, w, c, k; int32_t mode;
} rb_local_corr_warp_args;
int romab200_local_corr_warp(const rb_local_corr_warp_args* args, void* stream);

/* depthwise 5x5 conv (pad 2) + folded BN + ReLU on channels-last maps (create_block conv1+norm+relu,
 * matcher.py:106-120).  weight [25][ldw] fp32 (tap-major), bias [C] */
typedef struct {
    const void* in; void* out; int64_t ldi, ldo; const float* weight; int64_t ldw; const float* bias;
    int32_t batch, h, w, c; int32_t dtype;
    void* out_lo;   /* dtype == RB_F32 only: when non-NULL the result is written as an RB_F16S pair (out = hi plane, out_lo =
                       lo plane, pitch ldo in fp16 elements) so that the pointwise GEMM can consume it directly */
} rb_dwconv_args;
int romab200_dwconv5x5_relu(const rb_dwconv_args* args, void* stream);

/* Fused thin-map ConvRefiner block (C = 24, stride-1 maps): out = PW(ReLU(BN(DW5x5(in)))) in one pass.
 * in/out: channels-last 16-bit maps [batch, h, w, ld] (in != out); dw_weight [25][ldw] fp32 tap-major (BN folded), device.
 * pw_weight_host [c][c] fp32 row-major and pw_bias_host [c] are HOST arrays: the pointwise weights are passed to the
 * kernel as launch parameters (constant bank), they are read during this call only.  (create_block, matcher.py:92-122) */
typedef struct {
    const void* in; void* out; int64_t ld; const float* dw_weight; int64_t ldw; const float* dw_bias;
    const float* pw_weight_host; const float* pw_bias_host; int32_t batch, h, w, c; int32_t dtype;
} rb_refiner_block_small_args;
int romab200_refiner_block_small(const rb_refiner_block_small_args* args, void* stream);

/* Fused ConvRefiner block for the stride-2 maps (C = 144): depthwise 5x5 + BN + ReLU on the CUDA cores feeding a
 * tcgen05 pointwise GEMM whose weights stay resident in shared memory; one read + one write of the map.
 * in/out [batch, h, w, ld] (in != out); dw_weight [25][ldw] fp32 (BN folded).
 * dtype RB_F16 / RB_BF16: 16-bit maps, pw_weight [144][ld_pw] in the same type.
 * dtype RB_F32: fp32 maps (ld % 4 == 0, ldw even), pointwise weights as an RB_F16S pair: pw_weight = hi plane,
 * pw_weight_lo = lo plane, both [144][ld_pw] fp16.  The result is bit-identical to romab200_dwconv5x5_relu (RB_F32 in,
 * RB_F16S out) followed by the split-fp16 romab200_gemm with the pointwise bias. */
typedef struct {
    const void* in; void* out; int64_t ld; const float* dw_weight; int64_t ldw; const float* dw_bias;
    const void* pw_weight; int64_t ld_pw; const float* pw_bias; int32_t batch, h, w, c; int32_t dtype;
    const void* pw_weight_lo;   /* dtype == RB_F32 only */
} rb_refiner_block_c144_args;
int romab200_refiner_block_c144(const rb_refiner_block_c144_args* args, void* stream);

/* out_conv (fp32 1x1, C -> 3) + flow/certainty update (matcher.py:177-179, 496-506):
 * state[...,0] += scale_x * o0 ; state[...,1] += scale_y * o1 ; state[...,2] += o2 */
typedef struct {
    const void* d; int64_t ldd; const float* weight /* [3][ldw] */; int64_t ldw; const float* bias;
    float* state; int64_t rows; int32_t c; float scale_x, scale_y; int32_t dtype; float* delta_out /* optional [rows,3] */;
} rb_refiner_tail_args;
int romab200_refiner_tail(const rb_refiner_tail_args* args, void* stream);

/* bilinear resize, align_corners=False, no antialias (F.interpolate, matcher.py:424-435,513-523) of a
 * channels-last fp32 map [B, hi, wi, c] -> [B, ho, wo, c] */
typedef struct { const float* in; float* out; int32_t batch, hi, wi, ho, wo, c; } rb_resize_args;
int romab200_bilinear_resize(const rb_resize_args* args, void* stream);

/* match() epilogue (matcher.py:839-850, 891-927): certainty attenuation by the stride-16 logit, sigmoid,
 * out-of-range mask, clamp, identity grids and the symmetric concat.
 * state [D,H,W,3]; coarse_state [D,hc,wc,3] = the stride-16 state (NULL = no attenuation); warp [b,H,W*(sym?2:1),4]; cert [b,H,W*(sym?2:1)] */
typedef struct {
    const float* state; const float* coarse_state; int32_t hc, wc;
    float* warp; float* cert; int32_t b, H, W, symmetric;
    const float* grid_x; const float* grid_y;   /* pixel-centre linspaces of length W and H (matcher.py:904-912) */
} rb_match_epilogue_args;
int romab200_match_epilogue(const rb_match_epilogue_args* args, void* stream);

/* sample(): Gaussian KDE density (kde.py:4-12) without materialising the NxN matrix.
 * x [n,4] fp32; density[i] = sum_j exp(-||h(x_i)-h(x_j)||^2 / (2 std^2)), h = fp16 rounding when half != 0 */
typedef struct { const float* x; float* density; int32_t n; float std; int32_t half;
                 /* optional: workspace of splits * n floats; the j range is then cut into `splits` parts summed in a fixed order by a second
                  * kernel (more CTAs than SMs for the 40000-point problem of sample()).  NULL / splits <= 1: one pass */
                 float* workspace; int32_t splits;
                 /* half mode only: evaluate the block pairs (I, J >= I) of 256 x 256 points once and credit both the row and the column sums
                  * (exp(-d2) is symmetric); workspace of (splits + ceil(n / 256)) * n floats, its size in workspace_floats.  0: every pair twice */
                 int32_t symmetric; int64_t workspace_floats; } rb_kde_args;
int romab200_kde_density(const rb_kde_args* args, void* stream);

/* sample(): weighted sampling WITHOUT replacement on the device (the two torch.multinomial draws of matcher.py:613-617, 626-628).
 * For every batch item b: draws k distinct indices i in [0, n) with probabilities proportional to w_i = T(values[b*stride + i]),
 *   T = identity (RB_SAMPLE_IDENTITY), certainty thresholding `v > param ? 1 : v` (RB_SAMPLE_THRESHOLD, matcher.py:604-607), or density
 *   balancing `v < 10 ? 1e-7 : 1/(v+1)` of a KDE density v (RB_SAMPLE_BALANCE, matcher.py:622-625),
 * by an exponential race (key = -log(u)/w, k smallest keys; Philox4x32-10 keyed by `seed`, counter = element index).  out_idx [batch, k]
 * int32 in no particular order; out_weights (optional) [batch, k] receives the transformed weights of the drawn items; keys = workspace of
 * batch * n floats, scratch = workspace of batch * 2056 int32.  Items of zero weight are only drawn when fewer than k positive weights exist. */
enum rb_sample_transform { RB_SAMPLE_IDENTITY = 0, RB_SAMPLE_THRESHOLD = 1, RB_SAMPLE_BALANCE = 2 };
typedef struct {
    const float* values; int64_t n; int32_t k; int32_t batch; int64_t stride; uint64_t seed; int32_t transform; float param;
    int32_t* out_idx; float* out_weights; float* keys;
    void* scratch;   /* batch * 2056 * 4 bytes: histograms and selection state (cleared inside the call) */
    const uint64_t* seed_dev;   /* optional: the seed is read from this DEVICE word instead of `seed` (CUDA-graph replays with fresh seeds) */
} rb_sample_args;
int romab200_weighted_sample(const rb_sample_args* args, void* stream);

/* Image preprocessing in front of match() on the device: RGB uint8 image -> normalised fp32 [3, out_h, out_w]
 * (get_tuple_transform_ops(resize=(h, w), normalize=True), utils.py:164-173 = PIL.Image.resize((w, h), BICUBIC), /255, ImageNet mean/std;
 * called at matcher.py:812-815, 855-866).  Bit-exact with Pillow's 8-bit resampling (src/libImaging/Resample.c: 22-bit fixed-point weights,
 * horizontal pass into a uint8 image, then the vertical pass) and with the reference's fp32 operation order.
 *
 * romab200_resample_coeffs is HOST-ONLY arithmetic (no CUDA call, `stream` ignored): the weight table of one axis for in_size -> out_size,
 * bounds [out_size][2] = (first input sample, count), kk [out_size][ksize] zero-padded rows.  Call it with kk = bounds = NULL to get *ksize
 * first.  The tables depend on the two sizes only; keep device copies per size pair. */
typedef struct { int32_t in_size, out_size; int32_t* bounds; int32_t* kk; int32_t* ksize; } rb_resample_coeffs_args;
int romab200_resample_coeffs(const rb_resample_coeffs_args* args, void* stream);

typedef struct {
    const uint8_t* in; int64_t ld_in /* bytes per row */; int32_t in_h, in_w;   /* interleaved RGB, 3 bytes per pixel */
    int32_t out_h, out_w;
    const int32_t* bounds_x; const int32_t* kk_x; int32_t ksize_x;   /* DEVICE tables for in_w -> out_w (ignored when out_w == in_w) */
    const int32_t* bounds_y; const int32_t* kk_y; int32_t ksize_y;   /* DEVICE tables for in_h -> out_h (ignored when out_h == in_h) */
    uint8_t* tmp;      /* in_h * out_w * 3 bytes: the horizontally resampled image (unused when out_w == in_w) */
    uint8_t* out_u8;   /* optional [out_h, out_w, 3]: the resized 8-bit image, what PIL.Image.resize returns */
    float* out;        /* optional [3, out_h, out_w]: (u8 / 255 - mean) / std */
    float mean[3]; float std[3];
} rb_preprocess_args;
int romab200_preprocess_rgb8(const rb_preprocess_args* args, void* stream);

/* transpose a batched strided 2-D matrix: dst[b][c][r] = src[b][r][c]  (V^T for the PV product) */
typedef struct {
    const void* src; void* dst; int32_t rows, cols; int64_t lds, ldd; int32_t batch0, batch1;
    int64_t ss0, ss1, sd0, sd1; int32_t dtype;
} rb_transpose_args;
int romab200_transpose(const rb_transpose_args* args, void* stream);

/* debug: role-time counters of the tcgen05 GEMM kernels, collected when the environment variable ROMAB200_TC_CLK=1 is set before
 * the first GEMM (16 x uint64: MMA-thread / TMA-producer / epilogue wait and total cycles, tiles, k-blocks; scripts/gemm_clk.py) */
int romab200_debug_tc_clk(unsigned long long* out, int reset);

#ifdef __cplusplus
}
#endif
#endif /* ROMAB200_H */
