// tcgen05 / TMA GEMM back-end of romab200_gemm: fp16 / bf16 operands, fp32 accumulation in TMEM.
//
// One CTA computes one 128 x BN output tile (BN in {32, 64, 128, 256}).  Warp roles:
//   warp 0      TMA producer: one elected lane issues cp.async.bulk.tensor loads of the A (128 x 64) and
//               B (BN x 64, or 64 x BN when B is [K,N]) tiles into a STAGES-deep 128B-swizzled smem ring;
//   warp 1      allocates TMEM, then one elected lane issues tcgen05.mma (cta_group::1, kind::f16,
//               M=128, N=BN, K=16 per instruction, 4 per stage) and tcgen05.commit to free ring slots;
//   warps 2..5  epilogue: tcgen05.ld the fp32 accumulator (each warp owns the 32 TMEM lanes it may
//               address), apply the shared fused epilogue, store rows with 16-byte vector stores.
// A-operand "taps" (the 9 shifted row blocks of a 3x3 convolution on a zero-padded channels-last map) are
// just a per-k-block row offset on the TMA coordinate; out-of-range rows/columns are zero-filled by TMA,
// which also handles M/N/K tails, so no operand is ever padded or copied.
// Batched GEMMs (attention heads) use the 3rd/4th tensor-map dimension.
//
// SPLIT variant (dtype_ab == RB_F16S): fp32-class accuracy on the f16 tensor pipe.  Every operand element x is stored
// as two fp16 planes, hi = fp16(x) and lo = fp16((x - hi) * 2^11), i.e. 22 significand bits with the exponent range of
// fp16 and no underflow of the low part.  Per k-step the MMA thread issues three instructions into two TMEM
// accumulators, acc0 += A_hi.B_hi and acc1 += A_hi.B_lo + A_lo.B_hi; the epilogue forms acc0 + acc1 * 2^-11 (the
// dropped A_lo.B_lo term is 2^-22 relative).  Products of fp16 values are exact in the fp32 accumulator, so the only
// error left is the 2^-22 operand representation and the fp32 accumulation itself.
#include "common.cuh"
#include <cuda.h>

namespace rb {

// ------------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n" : "=r"(done) : "r"(addr), "r"(parity) : "memory");
    } while (!done);
}
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
// TMA stores (UTMASTG): shared -> global through a tensor map, tracked by bulk async-groups of the issuing thread
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
// the same as an element-wise fp32 reduction into global memory: C += tile (the in-place residual update)
__device__ __forceinline__ void tma_reduce_add_4d(const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2, int c3) {
    asm volatile("cp.reduce.async.bulk.tensor.4d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float* v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
          "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
          "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
          "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15])),
          "r"(__float_as_uint(v[16])), "r"(__float_as_uint(v[17])), "r"(__float_as_uint(v[18])), "r"(__float_as_uint(v[19])),
          "r"(__float_as_uint(v[20])), "r"(__float_as_uint(v[21])), "r"(__float_as_uint(v[22])), "r"(__float_as_uint(v[23])),
          "r"(__float_as_uint(v[24])), "r"(__float_as_uint(v[25])), "r"(__float_as_uint(v[26])), "r"(__float_as_uint(v[27])),
          "r"(__float_as_uint(v[28])), "r"(__float_as_uint(v[29])), "r"(__float_as_uint(v[30])), "r"(__float_as_uint(v[31]))
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 32 consecutive floats of a row vector (bias / LayerScale / residual): 8 x 16-byte loads when possible
__device__ __forceinline__ void load_row32(const float* __restrict__ p, float* out, bool full, int remaining) {
    if (full && (reinterpret_cast<uintptr_t>(p) & 15) == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            float4 t = reinterpret_cast<const float4*>(p)[j];
            out[4 * j] = t.x; out[4 * j + 1] = t.y; out[4 * j + 2] = t.z; out[4 * j + 3] = t.w;
        }
    } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) out[j] = j < remaining ? p[j] : 0.f;
    }
}

// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start>>4 | LBO>>4 <<16 | SBO>>4 <<32 | version 1 <<46 |
// layout SWIZZLE_128B (2) << 61
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// ------------------------------------------------------------------------------------------------
struct TcParams {
    int M, N, K;
    int batch1;
    int ntaps, k_per_tap; int tap_rows[9];
    int trans_b, is_bf16;
    int tiles_m, tiles_n, total_tiles;
    int64_t sc0, sc1, sr0, sr1, sna0, snb0;
    unsigned long long* clk;      // optional role-time counters (ROMAB200_TC_CLK=1): see tc_clk_dump
    int band_major;               // tile order: 1 = all N tiles of a row band before the next band, 0 = N-major (see tc_tile_coords)
    int epi_mode;                 // store strategy of the epilogue: 0 = direct row-per-lane stores, 2 = TMA stores from a per-warp staging
                                  // buffer (map_c / map_c_lo), 3 = the same as an fp32 reduce-add (C += tile)
    Epilogue epi;
};

// role-time instrumentation: cycles a role thread spent waiting / in total, summed over CTAs
//   [0] MMA wait full   [1] MMA wait tmem_empty   [2] MMA total   [3] producer wait empty   [4] producer total
//   [5] epilogue wait tmem_full (warp 2)   [6] epilogue total (warp 2)   [7] tiles (MMA thread)   [8] k-blocks
__device__ __forceinline__ void clk_add(unsigned long long* clk, int i, long long v) { if (clk) atomicAdd(&clk[i], (unsigned long long)v); }

constexpr int TC_BM = 128, TC_BK = 64;
constexpr int TC_STAGE_WORDS = 512;                // TMA-store staging buffer per epilogue warp: 32 rows x 64 bytes
constexpr int TC_PARK_WORDS = 1024;                // early-release park buffer per epilogue warp: one 32 x 32 fp32 chunk

template <int BN, bool SPLIT> struct TcCfg {
    // BN = 256: one CTA per SM with 8 epilogue warps; narrower tiles: two CTAs per SM (two MMA-issuing threads keep the
    // tensor pipe fed when a k-block is only 128-256 MMA cycles) with 4 epilogue warps each.  The split variant always
    // runs one CTA per SM (its two accumulators take up to all 512 TMEM columns).
    static constexpr int NOPS = SPLIT ? 2 : 1;                           // operand planes per matrix
    static constexpr int A_BYTES = TC_BM * TC_BK * 2;
    static constexpr int B_BYTES = BN * TC_BK * 2;
    static constexpr int STAGE_BYTES = NOPS * (A_BYTES + B_BYTES);
    static constexpr int STAGES = SPLIT ? (BN >= 144 ? 2 : (BN > 64 ? 3 : 4))
                                        : (BN >= 256 ? 4 : (BN > 128 ? 5 : (BN >= 128 ? 3 : 4)));
    static constexpr int CTAS_PER_SM = (SPLIT || BN > 128) ? 1 : 2;
    static constexpr int EPI_WARPS = BN > 128 ? 8 : 4;
    static constexpr int THREADS = 64 + 32 * EPI_WARPS;
    static constexpr int ACC_COLS = NOPS * BN;                           // TMEM columns of one accumulator stage
    static constexpr int ACC_STAGES = 2 * ACC_COLS <= 512 ? 2 : 1;       // double-buffered when it fits
    static constexpr bool EARLY = ACC_STAGES == 1 && BN <= 192;          // epilogue frees the accumulator before its math (tc_epilogue_tile)
    static constexpr int EPI_BYTES = 2 * 256 * 4 + EPI_WARPS * TC_STAGE_WORDS * 4 +  // staged bias / column-scale (or norm_b) + per-warp transpose buffers
                                     (EARLY ? EPI_WARPS * TC_PARK_WORDS * 4 : 0);    // + per-warp park buffers
    static constexpr int SMEM = STAGES * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/ + EPI_BYTES;
    static constexpr int ACC_TOTAL = ACC_STAGES * ACC_COLS;
    static constexpr int TMEM_COLS = ACC_TOTAL <= 32 ? 32 : (ACC_TOTAL <= 64 ? 64 : (ACC_TOTAL <= 128 ? 128 : (ACC_TOTAL <= 256 ? 256 : 512)));
    static_assert(SMEM <= 232448, "shared memory budget");
};

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// Tile index -> (m tile, n tile, batch index); the producer and the epilogue of both kernels decode through here.  Consecutive
// tiles run at about the same time on neighbouring CTAs, so the operand that the order keeps fixed is read from HBM once and shared
// in L2.  Band-major (the tiles_n tiles of a row band in a row) streams A once and re-reads B per band; N-major streams B once and
// re-reads A per N tile.  The host picks band-major when A is at least as large as B.
__device__ __forceinline__ void tc_tile_coords(const TcParams& p, int tile, int& mt, int& nt, int& z) {
    const int tiles_per_z = p.tiles_m * p.tiles_n;
    z = tile / tiles_per_z;
    const int r = tile - z * tiles_per_z;
    if (p.band_major) { mt = r / p.tiles_n; nt = r - mt * p.tiles_n; }
    else { nt = r / p.tiles_m; mt = r - nt * p.tiles_m; }
}

// Math and store of one 32-column chunk of the tile, held in v in the row-per-lane layout of tcgen05.ld (column cb of the tile).
__device__ __forceinline__ void tc_epilogue_chunk(const TcParams& p, const Epilogue& e, float (&v)[32], int cb, int m0, int n0, int z0, int z1, int q, int lane,
                                                  int nlim, int m, int64_t orow, bool vec_ok, const float* s_vec0, const float* s_vec1, float* stage,
                                                  const CUtensorMap* map_c, const CUtensorMap* map_c_lo, bool timing, int& t_math, int& t_store) {
    const int nb = n0 + cb;
    const long long tc1 = clock64();
    // ---- element-wise part in the row-per-lane layout (every branch is warp-uniform) ----
    if (e.epi == RB_EPI_COSKERNEL) {
        const float na = m < p.M ? e.norm_a[m] : 1.f;
        if (e.cos_normalized) {
            // operands are the L2-normalised rows: c = acc * pn / (pn + eps) = acc * (1 - eps / (pn + eps)).  eps / (pn + eps) is ~1e-9 of
            // the result, so an approximate reciprocal (2 ulp) leaves the factor correctly rounded in all but exotic cases (pn < 1e-2);
            // exp(x) = 2^(x log2 e) with x in [-2/T, 0]: the input rounding costs |x log2 e| 2^-24 < 1e-6 relative, an order below the
            // error of the split contraction itself (8e-6 vs float64).  15 instead of 30 instructions per element: this epilogue, not
            // the 8-k-block main loop, bounds the launch (ncu: tensor pipe 18 % active).
            const float k2 = e.inv_t * 1.4426950408889634f;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float4 b4 = *reinterpret_cast<const float4*>(&s_vec0[cb + 4 * j]);
                const float bn[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const float pe = fmaf(na, bn[t], e.eps);
                    float rc;
                    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc) : "f"(pe));
                    const float sc = fmaf(-e.eps, rc, 1.0f);
                    const float x2 = fmaf(v[4 * j + t], sc, -1.0f) * k2;
                    float r;
                    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x2));
                    v[4 * j + t] = r;
                }
            }
            if (e.diag_add != 0.f && m >= nb && m < nb + 32) {     // the diagonal crosses this 32-column chunk in at most one lane per column
#pragma unroll
                for (int j = 0; j < 32; ++j) if (m == nb + j) v[j] += e.diag_add;
            }
        } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const int n = nb + j;
                const float pn = na * s_vec0[cb + j];
                const float sc = 1.0f / (pn + e.eps);
                float r = expf((v[j] * sc - 1.0f) * e.inv_t);
                if (m == n) r += e.diag_add;
                v[j] = r;
            }
        }
    } else {
        if (e.alpha != 1.0f) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] *= e.alpha;
        }
        if (e.bias) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float4 b4 = *reinterpret_cast<const float4*>(&s_vec0[cb + 4 * j]);
                v[4 * j] += b4.x; v[4 * j + 1] += b4.y; v[4 * j + 2] += b4.z; v[4 * j + 3] += b4.w;
            }
        }
        if (e.act == RB_ACT_RELU) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
        } else if (e.act == RB_ACT_GELU) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = gelu_erf(v[j]);
        }
        if (e.col_scale) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float4 s4 = *reinterpret_cast<const float4*>(&s_vec1[cb + 4 * j]);
                v[4 * j] *= s4.x; v[4 * j + 1] *= s4.y; v[4 * j + 2] *= s4.z; v[4 * j + 3] *= s4.w;
            }
        }
    }
    // ---- store ----
    long long tc2 = clock64();
    t_math += (int)(tc2 - tc1);
    if (p.epi_mode >= 2) {
        // ---- TMA stores: the warp's 32 x 32 chunk goes through its 2 KB staging buffer as [32 rows][64 B] (16-bit output: one
        // round of 32 columns; fp32 / split pair: two rounds of 16 columns) and leaves with cp.async.bulk.tensor: whole segments,
        // clipped at the M / N tails by the tensor map, asynchronous to the warp.  Rows that are not stored (the zero border of a
        // padded map) are written as zeros, which is what they hold already.
        if (orow < 0) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = 0.f;
        }
        if (nb + 32 > nlim) {       // the N tail: TMA clips at 16-byte granules, so the pad columns up to the next granule receive zeros
#pragma unroll
            for (int j = 0; j < 32; ++j) if (nb + j >= nlim) v[j] = 0.f;
        }
        uint8_t* sb = reinterpret_cast<uint8_t*>(stage);
        const int row0 = m0 + q * 32;
        if (e.dtype_c == RB_F16 || e.dtype_c == RB_BF16) {
            if (lane == 0) bulk_wait_read();
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                uint32_t w[4];
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const float lo = v[8 * j + 2 * t], hi = v[8 * j + 2 * t + 1];
                    if (e.dtype_c == RB_F16) { __half2 hh = __floats2half2_rn(lo, hi); w[t] = *reinterpret_cast<uint32_t*>(&hh); }
                    else { __nv_bfloat162 hh = __floats2bfloat162_rn(lo, hi); w[t] = *reinterpret_cast<uint32_t*>(&hh); }
                }
                *reinterpret_cast<uint4*>(sb + lane * 64 + 16 * j) = make_uint4(w[0], w[1], w[2], w[3]);
            }
            fence_async_smem();
            __syncwarp();
            if (lane == 0) { tma_store_4d(map_c, sb, nb, row0, z1, z0); bulk_commit(); }
        } else {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                if (nb + 16 * h >= nlim) break;                 // warp-uniform
                if (lane == 0) bulk_wait_read();
                __syncwarp();
                if (e.dtype_c == RB_F32) {
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        *reinterpret_cast<float4*>(sb + lane * 64 + 16 * j) = make_float4(v[16 * h + 4 * j], v[16 * h + 4 * j + 1], v[16 * h + 4 * j + 2], v[16 * h + 4 * j + 3]);
                } else {                                        // RB_F16S: hi rows at [0, 1 KB), lo rows at [1 KB, 2 KB), 32 B each
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        uint32_t wh[4], wl[4];
#pragma unroll
                        for (int t = 0; t < 4; ++t) {
                            const float x0 = v[16 * h + 8 * j + 2 * t], x1 = v[16 * h + 8 * j + 2 * t + 1];
                            const __half2 hh = __floats2half2_rn(x0, x1);
                            const float2 hf = __half22float2(hh);
                            const __half2 ll = __floats2half2_rn((x0 - hf.x) * 2048.0f, (x1 - hf.y) * 2048.0f);
                            wh[t] = *reinterpret_cast<const uint32_t*>(&hh); wl[t] = *reinterpret_cast<const uint32_t*>(&ll);
                        }
                        *reinterpret_cast<uint4*>(sb + lane * 32 + 16 * j) = make_uint4(wh[0], wh[1], wh[2], wh[3]);
                        *reinterpret_cast<uint4*>(sb + 1024 + lane * 32 + 16 * j) = make_uint4(wl[0], wl[1], wl[2], wl[3]);
                    }
                }
                fence_async_smem();
                __syncwarp();
                if (lane == 0) {
                    if (e.dtype_c == RB_F32) {
                        if (p.epi_mode == 3) tma_reduce_add_4d(map_c, sb, nb + 16 * h, row0, z1, z0);
                        else tma_store_4d(map_c, sb, nb + 16 * h, row0, z1, z0);
                    } else {
                        tma_store_4d(map_c, sb, nb + 16 * h, row0, z1, z0);
                        tma_store_4d(map_c_lo, sb + 1024, nb + 16 * h, row0, z1, z0);
                    }
                    bulk_commit();
                }
            }
        }
    } else if (p.epi_mode == 0) {
        if (orow >= 0) {
        const bool full = nb + 32 <= nlim;
        if (e.epi != RB_EPI_COSKERNEL) {
        if (e.R) {
            if (e.dtype_r == RB_F32) {
                float rv[32];
                load_row32((const float*)e.R + orow * e.ldr + nb, rv, full, nlim - nb);
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] += rv[j];
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    if (nb + j < nlim) v[j] += load_any(e.R, orow * e.ldr + nb + j, e.dtype_r);
            }
        }
        }
    if (vec_ok) {
        if (e.dtype_c == RB_F32) {
            float* dst = (float*)e.C + orow * e.ldc + nb;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                if (nb + 4 * j + 4 <= nlim) *reinterpret_cast<float4*>(dst + 4 * j) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                else {
#pragma unroll
                    for (int t = 0; t < 4; ++t) if (nb + 4 * j + t < nlim) dst[4 * j + t] = v[4 * j + t];
                }
            }
        } else if (e.dtype_c == RB_F16S) {
            // split-pair output: hi = fp16(v), lo = fp16((v - hi) * 2^11) into two planes of the same pitch
            uint16_t* dhi = (uint16_t*)e.C + orow * e.ldc + nb;
            uint16_t* dlo = (uint16_t*)e.C_lo + orow * e.ldc + nb;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                uint32_t wh[4], wl[4];
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const float x0 = v[8 * j + 2 * t], x1 = v[8 * j + 2 * t + 1];
                    const __half2 h = __floats2half2_rn(x0, x1);
                    const float2 hf = __half22float2(h);
                    const __half2 l = __floats2half2_rn((x0 - hf.x) * 2048.0f, (x1 - hf.y) * 2048.0f);
                    wh[t] = *reinterpret_cast<const uint32_t*>(&h); wl[t] = *reinterpret_cast<const uint32_t*>(&l);
                }
                if (nb + 8 * j + 8 <= nlim) {
                    *reinterpret_cast<uint4*>(dhi + 8 * j) = make_uint4(wh[0], wh[1], wh[2], wh[3]);
                    *reinterpret_cast<uint4*>(dlo + 8 * j) = make_uint4(wl[0], wl[1], wl[2], wl[3]);
                } else {
#pragma unroll
                    for (int t = 0; t < 8; ++t)
                        if (nb + 8 * j + t < nlim) {
                            dhi[8 * j + t] = (uint16_t)(wh[t >> 1] >> (16 * (t & 1)));
                            dlo[8 * j + t] = (uint16_t)(wl[t >> 1] >> (16 * (t & 1)));
                        }
                }
            }
        } else {
            uint16_t* dst = (uint16_t*)e.C + orow * e.ldc + nb;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                uint32_t w[4];
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    float lo = v[8 * j + 2 * t], hi = v[8 * j + 2 * t + 1];
                    if (e.dtype_c == RB_F16) { __half2 h = __floats2half2_rn(lo, hi); w[t] = *reinterpret_cast<uint32_t*>(&h); }
                    else { __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi); w[t] = *reinterpret_cast<uint32_t*>(&h); }
                }
                if (nb + 8 * j + 8 <= nlim) *reinterpret_cast<uint4*>(dst + 8 * j) = make_uint4(w[0], w[1], w[2], w[3]);
                else {
#pragma unroll
                    for (int t = 0; t < 8; ++t)
                        if (nb + 8 * j + t < nlim) dst[8 * j + t] = (uint16_t)(w[t >> 1] >> (16 * (t & 1)));
                }
            }
        }
    } else {
#pragma unroll
        for (int j = 0; j < 32; ++j)
            if (nb + j < nlim) store_split_any(e.C, e.C_lo, orow * e.ldc + nb + j, e.dtype_c, v[j]);
    }
        }
    }
    __syncwarp();
    if (timing) { t_store += (int)(clock64() - tc2); }
}

// Epilogue of one 128 x BN accumulator tile by the EPI_WARPS epilogue warps of a CTA (shared by the 1-CTA and the 2-CTA
// kernels): stage the per-column vectors, wait for the accumulator, tcgen05.ld, fused epilogue, coalesced stores.
// `tmem_acc` = TMEM address of the tile's main accumulator (lane 0); the cross accumulator of the SPLIT variant sits BN columns
// further.  (m0, n0) = first row / column of the tile, z0 / z1 = batch indices.  `release()` gives the accumulator back to the MMA
// thread; EARLY (single-buffered 144 / 192-column split accumulators) calls it as soon as the warp's slice is out of the accumulator,
// otherwise after the stores.
//
// tcgen05.ld hands every lane ONE ROW of the accumulator, so a direct store writes 16-byte pieces of 32 different rows per
// instruction.  Measured with the role-time counters (ROMAB200_TC_CLK=1, scripts/gemm_clk.py) on the ViT shapes, cycles per
// 128 x 256 tile: store phase 6.1k (f16 out) / 11.6k (split pair out) against 8k / 25k cycles of MMA work; a shared-memory
// transpose to 4-lanes-per-row stores was slower still (12-15k: more instructions, the same line-granular L1 path).  So the
// tile leaves through the TMA unit instead: every warp writes its 32 x 32 chunk into a private 2 KB staging buffer as
// [32 rows][64 B] and one lane issues cp.async.bulk.tensor stores (UTMASTG; 3.3k / 5.6k cycles, asynchronous to the warp); an
// in-place fp32 residual (R == C) becomes a TMA reduce-add (UTMAREDG), so the residual stream is never read by the kernel.
// Row maps other than NONE / PAD_KEEP, mismatched residual operands and unaligned pitches take the direct path.
template <int BN, bool SPLIT, int EPI_WARPS, bool EARLY, class Release>
__device__ __forceinline__ void tc_epilogue_tile(const TcParams& p, uint32_t tmem_acc, uint64_t* full_bar, uint32_t full_parity, int m0, int n0,
                                                 int z0, int z1, int q, int half, int lane, int et, float* s_vec0, float* s_vec1, float* stage,
                                                 float* park, const CUtensorMap* map_c, const CUtensorMap* map_c_lo, Release release) {
    const long long t_entry = clock64();
    Epilogue e = p.epi;
    e.C = (char*)e.C + (z0 * p.sc0 + z1 * p.sc1) * dtype_size(e.dtype_c);
    if (e.C_lo) e.C_lo = (char*)e.C_lo + (z0 * p.sc0 + z1 * p.sc1) * 2;
    if (e.R) e.R = (const char*)e.R + (z0 * p.sr0 + z1 * p.sr1) * dtype_size(e.dtype_r);
    if (e.norm_a) e.norm_a += z0 * p.sna0;
    if (e.norm_b) e.norm_b += z0 * p.snb0;
    // stage the per-column epilogue vectors of this tile in shared memory (read back as broadcast float4s)
    asm volatile("bar.sync 1, %0;" ::"n"(32 * EPI_WARPS) : "memory");   // everyone is done with the previous tile's vectors
    for (int t = et; t < BN; t += 32 * EPI_WARPS) {
        const int n = n0 + t;
        const float* v0 = e.epi == RB_EPI_COSKERNEL ? e.norm_b : e.bias;
        s_vec0[t] = (v0 && n < p.N) ? v0[n] : (e.epi == RB_EPI_COSKERNEL ? 1.f : 0.f);
        s_vec1[t] = (e.col_scale && n < p.N) ? e.col_scale[n] : 1.f;
    }
    asm volatile("bar.sync 1, %0;" ::"n"(32 * EPI_WARPS) : "memory");
    const bool timing = p.clk && q == 2 && half == 0 && lane == 0;     // warp 2, lane 0
    const long long tw = clock64();
    const int t_pre = (int)(tw - t_entry);
    int t_ld = 0, t_math = 0, t_store = 0;              // cycles of this tile (warp 2, lane 0): fit 32 bits, spare registers
    mbar_wait(full_bar, full_parity);
    if (timing) clk_add(p.clk, 5, clock64() - tw);
    tc_fence_after();
    const int nlim = min(p.N, n0 + BN);                  // columns of this tile (BN need not be a multiple of 32)
    const int m = m0 + q * 32 + lane;
    const int64_t orow = m < p.M ? e.map_row(m) : -1;
    const int es_c = dtype_size(e.dtype_c);
    const bool vec_ok = (e.ldc * es_c) % 16 == 0 && (reinterpret_cast<uintptr_t>(e.C) % 16 == 0) &&
                        (e.dtype_c != RB_F16S || reinterpret_cast<uintptr_t>(e.C_lo) % 16 == 0);
    // one 32-column chunk of the accumulator (both accumulators of the SPLIT variant, combined); all 32 lanes take part in the TMEM
    // loads (.sync.aligned); rows that are not stored are masked in the store phase
    auto load_chunk = [&](int cb, float (&v)[32]) {
        tmem_ld32(tmem_acc + ((uint32_t)(q * 32) << 16) + cb, v);
        if constexpr (SPLIT) {
            float w[32];
            tmem_ld32(tmem_acc + ((uint32_t)(q * 32) << 16) + BN + cb, w);
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = fmaf(w[j], 1.0f / 2048.0f, v[j]);
        }
    };
    if constexpr (EARLY) {
        // single-buffered accumulator (split tiles of 144 / 192 columns): the warp first takes its whole row slice (at most 3 chunks of
        // 32 columns) out of the accumulator and gives it back, so that the math and the stores overlap the MMAs of the next tile.  The
        // combined chunks wait in TMEM columns the accumulator does not use (2 * BN .. 511: 64 per warp) and, the third one, in the
        // warp's 4 KB park buffer in shared memory.  (Holding them in registers spills: 10 warps leave 168 per thread.)  Park layout:
        // lane = row, its eight 16-byte granules XOR-swizzled by lane & 7, which keeps the accesses free of bank conflicts.
        constexpr int NCH = (BN + 8 * EPI_WARPS - 1) / (8 * EPI_WARPS);
        static_assert(NCH <= 3 && 2 * BN + 2 * 64 <= 512, "early release: two chunks per warp in spare TMEM columns, one in shared memory");
        const uint32_t spare = tmem_acc + ((uint32_t)(q * 32) << 16) + 2 * BN + half * 64;
        float4* prow = reinterpret_cast<float4*>(park) + lane * 8;
        const long long tc0 = clock64();
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
            const int cb = half * 32 + c * 8 * EPI_WARPS;
            if (cb < BN && n0 + cb < nlim) {                   // warp-uniform
                float v[32];
                load_chunk(cb, v);
                if (c < 2) {
                    tmem_st32(spare + 32 * c, v);
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j) prow[j ^ (lane & 7)] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                }
            }
        }
        tmem_st_wait();
        release();
        t_ld = (int)(clock64() - tc0);
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
            const int cb = half * 32 + c * 8 * EPI_WARPS;
            if (cb < BN && n0 + cb < nlim) {
                float v[32];
                if (c < 2) {
                    tmem_ld32(spare + 32 * c, v);
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float4 t = prow[j ^ (lane & 7)];
                        v[4 * j] = t.x; v[4 * j + 1] = t.y; v[4 * j + 2] = t.z; v[4 * j + 3] = t.w;
                    }
                }
                tc_epilogue_chunk(p, e, v, cb, m0, n0, z0, z1, q, lane, nlim, m, orow, vec_ok, s_vec0, s_vec1, stage, map_c, map_c_lo, timing, t_math, t_store);
            }
        }
    } else {
#pragma unroll 1
        for (int cb = half * 32; cb < BN; cb += 8 * EPI_WARPS) {
            if (n0 + cb >= nlim) break;                     // warp-uniform
            float v[32];
            const long long tc0 = clock64();
            load_chunk(cb, v);
            t_ld += (int)(clock64() - tc0);
            tc_epilogue_chunk(p, e, v, cb, m0, n0, z0, z1, q, lane, nlim, m, orow, vec_ok, s_vec0, s_vec1, stage, map_c, map_c_lo, timing, t_math, t_store);
        }
        release();
    }
    if (timing) { clk_add(p.clk, 11, t_pre); clk_add(p.clk, 12, t_ld); clk_add(p.clk, 13, t_math); clk_add(p.clk, 14, t_store); }
    __syncwarp();
}

// called by every epilogue warp before the CTA exits: the bulk stores it issued have completed
__device__ __forceinline__ void tc_epilogue_drain(const TcParams& p, int lane) {
    if (p.epi_mode >= 2 && lane == 0) bulk_wait_all();
    __syncwarp();
}

// Persistent kernel: every CTA walks tiles t = blockIdx.x, blockIdx.x + gridDim.x, ... in the order of tc_tile_coords (CTAs that
// run together share the larger operand's tiles in L2).  The accumulator is double-buffered in TMEM when it fits: the MMA warp
// starts the next tile while the epilogue warps drain the previous one.
template <int BN, bool SPLIT>
__global__ void __launch_bounds__(TcCfg<BN, SPLIT>::THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
               const __grid_constant__ CUtensorMap map_a_lo, const __grid_constant__ CUtensorMap map_b_lo,
               const __grid_constant__ CUtensorMap map_c, const __grid_constant__ CUtensorMap map_c_lo, const TcParams p) {
    using Cfg = TcCfg<BN, SPLIT>;
    constexpr int STAGES = Cfg::STAGES;
    constexpr int A_BYTES = Cfg::A_BYTES, B_BYTES = Cfg::B_BYTES;
    constexpr int OFF_A_LO = A_BYTES, OFF_B = Cfg::NOPS * A_BYTES, OFF_B_LO = Cfg::NOPS * A_BYTES + B_BYTES;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - ((uint32_t)__cvta_generic_to_shared(smem_raw) & 1023u)) & 1023u);   // offset on the array: keeps ld/st.shared
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::STAGE_BYTES);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tmem_full_bar = empty_bar + STAGES;       // [2]
    uint64_t* tmem_empty_bar = tmem_full_bar + 2;       // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);
    float* s_vec0 = reinterpret_cast<float*>(smem + STAGES * Cfg::STAGE_BYTES + 256);   // bias      | norm_b
    float* s_vec1 = s_vec0 + 256;                                                        // col_scale
    float* park = s_vec1 + 256 + Cfg::EPI_WARPS * TC_STAGE_WORDS + (threadIdx.x / 32 - 2) * TC_PARK_WORDS;   // this epilogue warp's (Cfg::EARLY)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int kblocks = (p.K + TC_BK - 1) / TC_BK;

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full_bar[s], 1); mbar_init(&tmem_empty_bar[s], Cfg::EPI_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // programmatic dependent launch: everything above (barrier init, TMEM allocation) overlapped the tail of the previous
    // kernel in the stream; its results may only be touched after this point
    rb::pdl_wait();

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            const int kb_per_tap = p.ntaps > 1 ? p.k_per_tap / TC_BK : kblocks;
            uint32_t it = 0;
            long long w_empty = 0; const long long t_begin = clock64();
            for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
                int mt, nt, z;
                tc_tile_coords(p, tile, mt, nt, z);
                const int m0 = mt * TC_BM, n0 = nt * BN, z0 = z / p.batch1, z1 = z - z0 * p.batch1;
                for (int kb = 0; kb < kblocks; ++kb, ++it) {
                    const int s = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    const long long tw = clock64();
                    mbar_wait(&empty_bar[s], ph ^ 1);
                    w_empty += clock64() - tw;
                    mbar_expect_tx(&full_bar[s], Cfg::STAGE_BYTES);
                    int tap = 0, kin = kb * TC_BK, shift = 0;
                    if (p.ntaps > 1) { tap = kb / kb_per_tap; kin = (kb - tap * kb_per_tap) * TC_BK; shift = p.tap_rows[tap]; }
                    uint8_t* st = smem + s * Cfg::STAGE_BYTES;
                    tma_load_4d(st, &map_a, &full_bar[s], kin, m0 + shift, z1, z0);
                    if constexpr (SPLIT) tma_load_4d(st + OFF_A_LO, &map_a_lo, &full_bar[s], kin, m0 + shift, z1, z0);
                    if (!p.trans_b) {
                        tma_load_4d(st + OFF_B, &map_b, &full_bar[s], kb * TC_BK, n0, z1, z0);
                        if constexpr (SPLIT) tma_load_4d(st + OFF_B_LO, &map_b_lo, &full_bar[s], kb * TC_BK, n0, z1, z0);
                    } else {
                        // B is [K, N]: boxes of 64 (n) x 64 (k); one box per 64 columns of the tile
#pragma unroll
                        for (int j = 0; j < (BN + 63) / 64; ++j) {
                            tma_load_4d(st + OFF_B + j * (64 * 128), &map_b, &full_bar[s], n0 + j * 64, kb * TC_BK, z1, z0);
                            if constexpr (SPLIT) tma_load_4d(st + OFF_B_LO + j * (64 * 128), &map_b_lo, &full_bar[s], n0 + j * 64, kb * TC_BK, z1, z0);
                        }
                    }
                }
            }
            clk_add(p.clk, 3, w_empty); clk_add(p.clk, 4, clock64() - t_begin);
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            // instruction descriptor: D=f32, A/B = f16|bf16, A K-major, B K-major or MN-major, N>>3, M>>4
            uint32_t idesc = 0;
            idesc |= 1u << 4;
            idesc |= (uint32_t)(p.is_bf16 ? 1 : 0) << 7;
            idesc |= (uint32_t)(p.is_bf16 ? 1 : 0) << 10;
            idesc |= (uint32_t)(p.trans_b ? 1 : 0) << 16;
            idesc |= (uint32_t)(BN >> 3) << 17;
            idesc |= (uint32_t)(TC_BM >> 4) << 24;
            uint32_t it = 0, tcount = 0;
            long long w_full = 0, w_tmem = 0; const long long t_begin = clock64();
            for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++tcount) {
                const uint32_t acc = tcount % Cfg::ACC_STAGES, acc_ph = (tcount / Cfg::ACC_STAGES) & 1;
                long long tw = clock64();
                mbar_wait(&tmem_empty_bar[acc], acc_ph ^ 1);          // epilogue has drained this accumulator
                w_tmem += clock64() - tw;
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + acc * Cfg::ACC_COLS;
                for (int kb = 0; kb < kblocks; ++kb, ++it) {
                    const int s = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    tw = clock64();
                    mbar_wait(&full_bar[s], ph);
                    w_full += clock64() - tw;
                    tc_fence_after();
                    const uint32_t st = smem_u32(smem + s * Cfg::STAGE_BYTES);
                    // k-steps that lie entirely beyond K hold TMA zero fill only: skip them (K = 24, 144, 1377 ...)
                    const int krem = p.ntaps > 1 ? TC_BK : p.K - kb * TC_BK;        // taps are whole k-blocks
                    const int ksteps = krem >= TC_BK ? TC_BK / 16 : (krem + 15) / 16;
#pragma unroll
                    for (int k = 0; k < TC_BK / 16; ++k) {
                        if (k < ksteps) {
                            // K-major SW128: 8-row groups are 1024 B apart (SBO); a K step of 16 elements = +32 B inside the atom
                            const uint32_t koff_a = k * 32, koff_b = p.trans_b ? k * 2048 : k * 32;   // MN-major B: +2 k-groups
                            const uint32_t lbo_b = p.trans_b ? 64 * 128 : 16;
                            const uint64_t a_hi = make_smem_desc(st + koff_a, 16, 1024);
                            const uint64_t b_hi = make_smem_desc(st + OFF_B + koff_b, lbo_b, 1024);
                            const uint32_t accum = (kb | k) != 0;
                            umma_f16(tmem_d, a_hi, b_hi, idesc, accum);
                            if constexpr (SPLIT) {
                                const uint64_t a_lo = make_smem_desc(st + OFF_A_LO + koff_a, 16, 1024);
                                const uint64_t b_lo = make_smem_desc(st + OFF_B_LO + koff_b, lbo_b, 1024);
                                umma_f16(tmem_d + BN, a_hi, b_lo, idesc, accum);
                                umma_f16(tmem_d + BN, a_lo, b_hi, idesc, 1u);
                            }
                        }
                    }
                    umma_commit(&empty_bar[s]);          // frees the smem slot when these MMAs retire
                }
                umma_commit(&tmem_full_bar[acc]);        // accumulator complete
            }
            clk_add(p.clk, 0, w_full); clk_add(p.clk, 1, w_tmem); clk_add(p.clk, 2, clock64() - t_begin);
            clk_add(p.clk, 7, tcount); clk_add(p.clk, 8, it);
        }
    } else {
        // ===== epilogue (warps 2..9): TMEM lane quarter = warp % 4; the two warps of a quarter split the column chunks =====
        const int q = warp & 3;
        const int half = (warp - 2) >> 2;
        const int et = threadIdx.x - 64;                      // 0..255 among the epilogue threads
        uint32_t tcount = 0;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++tcount) {
            int mt, nt, z;
            tc_tile_coords(p, tile, mt, nt, z);
            const int m0 = mt * TC_BM, n0 = nt * BN, z0 = z / p.batch1, z1 = z - z0 * p.batch1;
            const uint32_t acc = tcount % Cfg::ACC_STAGES, acc_ph = (tcount / Cfg::ACC_STAGES) & 1;
            const long long te = clock64();
            auto release = [&] { tc_fence_before(); __syncwarp(); if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]); };
            tc_epilogue_tile<BN, SPLIT, Cfg::EPI_WARPS, Cfg::EARLY>(p, tmem_base + acc * Cfg::ACC_COLS, &tmem_full_bar[acc], acc_ph, m0, n0, z0, z1, q, half, lane, et,
                                                                  s_vec0, s_vec1, s_vec1 + 256 + (warp - 2) * TC_STAGE_WORDS, park, &map_c, &map_c_lo, release);
            if (warp == 2 && lane == 0) clk_add(p.clk, 6, clock64() - te);
        }
        tc_epilogue_drain(p, lane);
    }
    __syncthreads();
    if (warp == 1) { tc_fence_after(); tmem_dealloc(tmem_base, Cfg::TMEM_COLS); }
}


// ------------------------------------------------------------------------------------------------
// CTA-pair (cta_group::2) primitives.  Within a cluster the 32-bit shared-window address carries the CTA rank in bit 24
// (cute::Sm100MmaPeerBitMask), so clearing that bit turns a local barrier address into the leader's (rank 0) barrier.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_load_4d_pair(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
    // executed by both CTAs of the pair: the bytes land in the caller's shared memory, the transaction count on the LEADER's barrier
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_slot, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives (once the MMAs issued so far have retired) on the barrier at this shared-memory offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
    const uint16_t mask = 3;
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)), "h"(mask) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cta(uint64_t* bar, uint32_t cta) {     // arrive on `bar` of CTA `cta` of the cluster
    asm volatile(
        "{\n"
        ".reg .b32 ra;\n"
        "mapa.shared::cluster.u32 ra, %0, %1;\n"
        "mbarrier.arrive.shared::cluster.b64 _, [ra];\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(cta) : "memory");
}

template <int BN, bool SPLIT> struct TcPairCfg {
    // CTA pair = one 256 x BN tile: each CTA holds 128 rows of A and BN/2 rows of B per k-block (half the B traffic of two
    // independent 128 x BN tiles) and its own 128 x BN accumulator rows in TMEM.
    static constexpr int NOPS = SPLIT ? 2 : 1;
    static constexpr int A_BYTES = TC_BM * TC_BK * 2;
    static constexpr int B_BYTES = (BN / 2) * TC_BK * 2;                 // this CTA's half of the B tile
    static constexpr int STAGE_BYTES = NOPS * (A_BYTES + B_BYTES);
    static constexpr int EPI_WARPS = 8;
    static constexpr int VEC_BYTES = 2 * 256 * 4 + EPI_WARPS * TC_STAGE_WORDS * 4;
    static constexpr int STAGES = (232448 - 1024 - 256 - VEC_BYTES) / STAGE_BYTES > 6 ? 6 : (232448 - 1024 - 256 - VEC_BYTES) / STAGE_BYTES;
    static constexpr int THREADS = 64 + 32 * EPI_WARPS;
    static constexpr int ACC_COLS = NOPS * BN;
    static constexpr int ACC_STAGES = 2 * ACC_COLS <= 512 ? 2 : 1;
    static constexpr int ACC_TOTAL = ACC_STAGES * ACC_COLS;
    static constexpr int TMEM_COLS = ACC_TOTAL <= 256 ? 256 : 512;
    // early release (tc_epilogue_tile) needs spare TMEM columns and a 4 KB park buffer per epilogue warp: 192 has both, 256 neither
    static constexpr bool EARLY = ACC_STAGES == 1 && BN <= 192;
    static constexpr int EPI_BYTES = VEC_BYTES + (EARLY ? EPI_WARPS * TC_PARK_WORDS * 4 : 0);
    static constexpr int SMEM = STAGES * STAGE_BYTES + 1024 + 256 + EPI_BYTES;
    static_assert(BN % 32 == 0 && BN <= 256 && STAGES >= 2, "pair tile");
    static_assert(SMEM <= 232448, "shared memory budget");
};

// Persistent CTA-pair kernel: cluster c walks pair tiles t = c, c + #clusters, ...  Rank 0 (the leader) issues every MMA
// (tcgen05.mma.cta_group::2, M = 256); both CTAs run a TMA producer (own A rows, own half of B, signalling the leader's full
// barrier) and epilogue warps (own 128 accumulator rows).  Barriers: full[s] leader only (armed with the bytes of both CTAs);
// empty[s] and tmem_full[a] in both CTAs, released by multicast commits; tmem_empty[a] leader only, 2 x EPI_WARPS arrivals.
template <int BN, bool SPLIT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TcPairCfg<BN, SPLIT>::THREADS, 1)
gemm_tc_pair_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                    const __grid_constant__ CUtensorMap map_a_lo, const __grid_constant__ CUtensorMap map_b_lo,
                    const __grid_constant__ CUtensorMap map_c, const __grid_constant__ CUtensorMap map_c_lo, const TcParams p) {
    using Cfg = TcPairCfg<BN, SPLIT>;
    constexpr int STAGES = Cfg::STAGES;
    constexpr int A_BYTES = Cfg::A_BYTES, B_BYTES = Cfg::B_BYTES;
    constexpr int OFF_A_LO = A_BYTES, OFF_B = Cfg::NOPS * A_BYTES, OFF_B_LO = Cfg::NOPS * A_BYTES + B_BYTES;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - ((uint32_t)__cvta_generic_to_shared(smem_raw) & 1023u)) & 1023u);   // offset on the array: keeps ld/st.shared
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::STAGE_BYTES);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tmem_full_bar = empty_bar + STAGES;       // [2]
    uint64_t* tmem_empty_bar = tmem_full_bar + 2;       // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);
    float* s_vec0 = reinterpret_cast<float*>(smem + STAGES * Cfg::STAGE_BYTES + 256);
    float* s_vec1 = s_vec0 + 256;
    float* park = s_vec1 + 256 + Cfg::EPI_WARPS * TC_STAGE_WORDS + (threadIdx.x / 32 - 2) * TC_PARK_WORDS;   // this epilogue warp's (Cfg::EARLY)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const int cid = blockIdx.x >> 1, nclusters = gridDim.x >> 1;
    const int kblocks = (p.K + TC_BK - 1) / TC_BK;

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full_bar[s], 1); mbar_init(&tmem_empty_bar[s], 2 * Cfg::EPI_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc_pair(tmem_slot, Cfg::TMEM_COLS);
    tc_fence_before();
    cluster_sync_all();                 // both CTAs' barriers are initialised before anything signals across the pair
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    rb::pdl_wait();

    if (warp == 0) {
        // ===== TMA producer (both CTAs) =====
        if (lane == 0) {
            const int kb_per_tap = p.ntaps > 1 ? p.k_per_tap / TC_BK : kblocks;
            uint32_t it = 0;
            long long w_empty = 0; const long long t_begin = clock64();
            for (int tile = cid; tile < p.total_tiles; tile += nclusters) {
                int mt, nt, z;
                tc_tile_coords(p, tile, mt, nt, z);
                const int m0 = mt * (2 * TC_BM) + (int)rank * TC_BM, n0 = nt * BN + (int)rank * (BN / 2);
                const int z0 = z / p.batch1, z1 = z - z0 * p.batch1;
                for (int kb = 0; kb < kblocks; ++kb, ++it) {
                    const int s = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    const long long tw = clock64();
                    mbar_wait(&empty_bar[s], ph ^ 1);
                    w_empty += clock64() - tw;
                    if (rank == 0) mbar_expect_tx(&full_bar[s], 2 * Cfg::STAGE_BYTES);
                    int tap = 0, kin = kb * TC_BK, shift = 0;
                    if (p.ntaps > 1) { tap = kb / kb_per_tap; kin = (kb - tap * kb_per_tap) * TC_BK; shift = p.tap_rows[tap]; }
                    uint8_t* st = smem + s * Cfg::STAGE_BYTES;
                    tma_load_4d_pair(st, &map_a, &full_bar[s], kin, m0 + shift, z1, z0);
                    if constexpr (SPLIT) tma_load_4d_pair(st + OFF_A_LO, &map_a_lo, &full_bar[s], kin, m0 + shift, z1, z0);
                    tma_load_4d_pair(st + OFF_B, &map_b, &full_bar[s], kb * TC_BK, n0, z1, z0);
                    if constexpr (SPLIT) tma_load_4d_pair(st + OFF_B_LO, &map_b_lo, &full_bar[s], kb * TC_BK, n0, z1, z0);
                }
            }
            clk_add(p.clk, rank ? 9 : 3, w_empty); clk_add(p.clk, rank ? 10 : 4, clock64() - t_begin);
        }
    } else if (warp == 1) {
        // ===== MMA issuer (leader CTA only) =====
        if (rank == 0 && lane == 0) {
            // instruction descriptor: D=f32, A/B = f16|bf16 K-major, N>>3, M = 256 >> 4
            uint32_t idesc = 0;
            idesc |= 1u << 4;
            idesc |= (uint32_t)(p.is_bf16 ? 1 : 0) << 7;
            idesc |= (uint32_t)(p.is_bf16 ? 1 : 0) << 10;
            idesc |= (uint32_t)(BN >> 3) << 17;
            idesc |= (uint32_t)((2 * TC_BM) >> 4) << 24;
            uint32_t it = 0, tcount = 0;
            long long w_full = 0, w_tmem = 0; const long long t_begin = clock64();
            for (int tile = cid; tile < p.total_tiles; tile += nclusters, ++tcount) {
                const uint32_t acc = tcount % Cfg::ACC_STAGES, acc_ph = (tcount / Cfg::ACC_STAGES) & 1;
                long long tw = clock64();
                mbar_wait(&tmem_empty_bar[acc], acc_ph ^ 1);          // both CTAs' epilogues have drained this accumulator
                w_tmem += clock64() - tw;
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + acc * Cfg::ACC_COLS;
                for (int kb = 0; kb < kblocks; ++kb, ++it) {
                    const int s = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    tw = clock64();
                    mbar_wait(&full_bar[s], ph);
                    w_full += clock64() - tw;
                    tc_fence_after();
                    const uint32_t st = smem_u32(smem + s * Cfg::STAGE_BYTES);
                    const int krem = p.ntaps > 1 ? TC_BK : p.K - kb * TC_BK;
                    const int ksteps = krem >= TC_BK ? TC_BK / 16 : (krem + 15) / 16;
#pragma unroll
                    for (int k = 0; k < TC_BK / 16; ++k) {
                        if (k < ksteps) {
                            const uint64_t a_hi = make_smem_desc(st + k * 32, 16, 1024);
                            const uint64_t b_hi = make_smem_desc(st + OFF_B + k * 32, 16, 1024);
                            const uint32_t accum = (kb | k) != 0;
                            umma_f16_pair(tmem_d, a_hi, b_hi, idesc, accum);
                            if constexpr (SPLIT) {
                                const uint64_t a_lo = make_smem_desc(st + OFF_A_LO + k * 32, 16, 1024);
                                const uint64_t b_lo = make_smem_desc(st + OFF_B_LO + k * 32, 16, 1024);
                                umma_f16_pair(tmem_d + BN, a_hi, b_lo, idesc, accum);
                                umma_f16_pair(tmem_d + BN, a_lo, b_hi, idesc, 1u);
                            }
                        }
                    }
                    umma_commit_pair(&empty_bar[s]);          // frees the smem slot in both CTAs when these MMAs retire
                }
                umma_commit_pair(&tmem_full_bar[acc]);        // accumulator complete (both CTAs' epilogues)
            }
            clk_add(p.clk, 0, w_full); clk_add(p.clk, 1, w_tmem); clk_add(p.clk, 2, clock64() - t_begin);
            clk_add(p.clk, 7, tcount); clk_add(p.clk, 8, it);
        }
    } else {
        // ===== epilogue (warps 2..9, both CTAs): this CTA's 128 rows of the pair tile =====
        const int q = warp & 3;
        const int half = (warp - 2) >> 2;
        const int et = threadIdx.x - 64;
        uint32_t tcount = 0;
        for (int tile = cid; tile < p.total_tiles; tile += nclusters, ++tcount) {
            int mt, nt, z;
            tc_tile_coords(p, tile, mt, nt, z);
            const int m0 = mt * (2 * TC_BM) + (int)rank * TC_BM, n0 = nt * BN, z0 = z / p.batch1, z1 = z - z0 * p.batch1;
            const uint32_t acc = tcount % Cfg::ACC_STAGES, acc_ph = (tcount / Cfg::ACC_STAGES) & 1;
            const long long te = clock64();
            auto release = [&] { tc_fence_before(); __syncwarp(); if (lane == 0) mbar_arrive_cta(&tmem_empty_bar[acc], 0); };
            tc_epilogue_tile<BN, SPLIT, Cfg::EPI_WARPS, Cfg::EARLY>(p, tmem_base + acc * Cfg::ACC_COLS, &tmem_full_bar[acc], acc_ph, m0, n0, z0, z1, q, half, lane, et,
                                                                  s_vec0, s_vec1, s_vec1 + 256 + (warp - 2) * TC_STAGE_WORDS, park, &map_c, &map_c_lo, release);
            if (warp == 2 && lane == 0 && rank == 0) clk_add(p.clk, 6, clock64() - te);
        }
        tc_epilogue_drain(p, lane);
    }
    tc_fence_before();
    cluster_sync_all();                 // the peer's shared memory and barriers stay valid until the leader's last MMA / commit
    if (warp == 1) { tc_fence_after(); tmem_dealloc_pair(tmem_base, Cfg::TMEM_COLS); }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) != cudaSuccess || !ptr) return nullptr;
        fn = (EncodeTiledFn)ptr;
    }
    return fn;
}

// 4-D map over (columns, rows, batch1, batch0) of an OUTPUT matrix for the TMA-store epilogue: no swizzle, box = box_cols x 32 rows
static int make_out_map(CUtensorMap* map, void* base, int dtype, uint64_t cols, uint64_t rows, uint64_t pitch_elems, uint64_t b1, uint64_t s1_elems,
                        uint64_t b0, uint64_t s0_elems, uint32_t box_cols);

// 4-D map over (inner, rows, batch1, batch0) of a 16-bit matrix
static int make_map(CUtensorMap* map, const void* base, int is_bf16, uint64_t inner, uint64_t rows, uint64_t pitch_elems, uint64_t b1,
                    uint64_t s1_elems, uint64_t b0, uint64_t s0_elems, uint32_t box_inner, uint32_t box_rows) {
    EncodeTiledFn enc = get_encode();
    RB_REQUIRE(enc, "gemm_tc: cuTensorMapEncodeTiled not available (driver too old?)");
    RB_REQUIRE(((uintptr_t)base) % 16 == 0 && (pitch_elems * 2) % 16 == 0, "gemm_tc: operand base/pitch must be 16-byte aligned (pitch %llu elems)", (unsigned long long)pitch_elems);
    RB_REQUIRE((b1 <= 1 || (s1_elems * 2) % 16 == 0) && (b0 <= 1 || (s0_elems * 2) % 16 == 0), "gemm_tc: batch strides must be 16-byte aligned");
    cuuint64_t dims[4] = {inner, rows, b1 > 0 ? b1 : 1, b0 > 0 ? b0 : 1};
    cuuint64_t strides[3] = {pitch_elems * 2, (b1 > 1 ? s1_elems : pitch_elems * rows) * 2, (b0 > 1 ? s0_elems : pitch_elems * rows) * 2};
    cuuint32_t box[4] = {box_inner, box_rows, 1, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(map, is_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(base), dims,
                     strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    RB_REQUIRE(r == CUDA_SUCCESS, "gemm_tc: cuTensorMapEncodeTiled failed with %d (inner=%llu rows=%llu pitch=%llu)", (int)r,
               (unsigned long long)inner, (unsigned long long)rows, (unsigned long long)pitch_elems);
    return 0;
}

static int make_out_map(CUtensorMap* map, void* base, int dtype, uint64_t cols, uint64_t rows, uint64_t pitch_elems, uint64_t b1, uint64_t s1_elems,
                        uint64_t b0, uint64_t s0_elems, uint32_t box_cols) {
    EncodeTiledFn enc = get_encode();
    RB_REQUIRE(enc, "gemm_tc: cuTensorMapEncodeTiled not available (driver too old?)");
    const uint64_t es = dtype == RB_F32 ? 4 : 2;
    cuuint64_t dims[4] = {cols, rows, b1 > 0 ? b1 : 1, b0 > 0 ? b0 : 1};
    cuuint64_t strides[3] = {pitch_elems * es, (b1 > 1 ? s1_elems : pitch_elems * rows) * es, (b0 > 1 ? s0_elems : pitch_elems * rows) * es};
    cuuint32_t box[4] = {box_cols, 32, 1, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    const CUtensorMapDataType dt = dtype == RB_F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : (dtype == RB_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16);
    CUresult r = enc(map, dt, 4, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                     CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    RB_REQUIRE(r == CUDA_SUCCESS, "gemm_tc: cuTensorMapEncodeTiled (output) failed with %d (cols=%llu rows=%llu pitch=%llu)", (int)r,
               (unsigned long long)cols, (unsigned long long)rows, (unsigned long long)pitch_elems);
    return 0;
}

struct TcMaps { CUtensorMap a, b, a_lo, b_lo, c, c_lo; };

static unsigned long long* tc_clk_buffer() {        // ROMAB200_TC_CLK=1: role-time counters in a device buffer (debug)
    static unsigned long long* buf = nullptr;
    static int init = 0;
    if (!init) {
        init = 1;
        const char* e = getenv("ROMAB200_TC_CLK");
        if (e && atoi(e)) { if (cudaMalloc(&buf, 16 * sizeof(unsigned long long)) != cudaSuccess) buf = nullptr; else cudaMemset(buf, 0, 16 * sizeof(unsigned long long)); }
    }
    return buf;
}

static int sm_count() {
    static int n[64] = {};
    const int dev = current_device() & 63;
    if (!n[dev]) {
        cudaDeviceGetAttribute(&n[dev], cudaDevAttrMultiProcessorCount, dev);
        if (n[dev] <= 0) n[dev] = 148;
    }
    return n[dev];
}

static thread_local int g_max_ctas = 0;       // rb_gemm_args.max_ctas of the call being launched (0: no cap)

template <int BN, bool SPLIT>
static int launch_tc(const TcMaps& maps, TcParams& p, int zdim, cudaStream_t st) {
    using Cfg = TcCfg<BN, SPLIT>;
    // function attributes are per device: one flag per device ordinal (several engines on different GPUs in one process)
    static bool configured[64] = {};
    const int dev = current_device();
    if (!configured[dev & 63]) {
        cudaError_t e = cudaFuncSetAttribute(gemm_tc_kernel<BN, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM);
        RB_REQUIRE(e == cudaSuccess, "gemm_tc: cannot set %d bytes of dynamic shared memory: %s", Cfg::SMEM, cudaGetErrorString(e));
        configured[dev & 63] = true;
    }
    p.tiles_m = (p.M + TC_BM - 1) / TC_BM;
    p.tiles_n = (p.N + BN - 1) / BN;
    const long long total = (long long)p.tiles_m * p.tiles_n * zdim;
    RB_REQUIRE(total < (1ll << 31), "gemm_tc: too many tiles");
    p.total_tiles = (int)total;
    int resident = sm_count() * Cfg::CTAS_PER_SM;
    if (g_max_ctas > 0 && g_max_ctas < resident) resident = g_max_ctas;
    const int grid = p.total_tiles < resident ? p.total_tiles : resident;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(Cfg::THREADS); cfg.dynamicSmemBytes = Cfg::SMEM; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = rb::pdl_mode() == 1 ? 0 : 1;
    cudaError_t err = cudaLaunchKernelEx(&cfg, gemm_tc_kernel<BN, SPLIT>, maps.a, maps.b, maps.a_lo, maps.b_lo, maps.c, maps.c_lo, (const TcParams)p);
    if (err != cudaSuccess) { set_error("gemm_tc: launch failed: %s", cudaGetErrorString(err)); return 1; }
    return check_launch("gemm_tc");
}

// 0: never, 1 (default): when profitable, 2: whenever legal (tests).  Environment variable ROMAB200_GEMM_PAIR.
static int wave_rule() { static const int m = [] { const char* e = getenv("ROMAB200_GEMM_WAVE"); return e ? atoi(e) : 1; }(); return m; }
static int pair_mode() { static const int m = [] { const char* e = getenv("ROMAB200_GEMM_PAIR"); return e ? atoi(e) : 1; }(); return m; }

template <int BN, bool SPLIT>
static int launch_tc_pair(const TcMaps& maps, TcParams& p, int zdim, cudaStream_t st) {
    using Cfg = TcPairCfg<BN, SPLIT>;
    static bool configured[64] = {};
    const int dev = current_device();
    if (!configured[dev & 63]) {
        cudaError_t e = cudaFuncSetAttribute(gemm_tc_pair_kernel<BN, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM);
        RB_REQUIRE(e == cudaSuccess, "gemm_tc(pair): cannot set %d bytes of dynamic shared memory: %s", Cfg::SMEM, cudaGetErrorString(e));
        configured[dev & 63] = true;
    }
    p.tiles_m = (p.M + 2 * TC_BM - 1) / (2 * TC_BM);
    p.tiles_n = (p.N + BN - 1) / BN;
    const long long total = (long long)p.tiles_m * p.tiles_n * zdim;
    RB_REQUIRE(total < (1ll << 31), "gemm_tc: too many tiles");
    p.total_tiles = (int)total;
    int pairs = sm_count() / 2;
    if (g_max_ctas > 1 && g_max_ctas / 2 < pairs) pairs = g_max_ctas / 2;
    const int nclusters = p.total_tiles < pairs ? p.total_tiles : pairs;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * nclusters); cfg.blockDim = dim3(Cfg::THREADS); cfg.dynamicSmemBytes = Cfg::SMEM; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = rb::pdl_mode() == 1 ? 0 : 1;
    cudaError_t err = cudaLaunchKernelEx(&cfg, gemm_tc_pair_kernel<BN, SPLIT>, maps.a, maps.b, maps.a_lo, maps.b_lo, maps.c, maps.c_lo, (const TcParams)p);
    if (err != cudaSuccess) { set_error("gemm_tc(pair): launch failed: %s", cudaGetErrorString(err)); return 1; }
    return check_launch("gemm_tc_pair");
}

template <bool SPLIT>
static int dispatch_tc(int BN, const TcMaps& maps, TcParams& p, int zdim, cudaStream_t st) {
    switch (BN) {
        case 32: return launch_tc<32, SPLIT>(maps, p, zdim, st);
        case 64: return launch_tc<64, SPLIT>(maps, p, zdim, st);
        case 128: return launch_tc<128, SPLIT>(maps, p, zdim, st);
        case 144: return launch_tc<144, SPLIT>(maps, p, zdim, st);
        case 192: return launch_tc<192, SPLIT>(maps, p, zdim, st);
        default: return launch_tc<256, SPLIT>(maps, p, zdim, st);
    }
}

int gemm_tc(const rb_gemm_args* a, cudaStream_t stream) {
    RB_REQUIRE(a->dtype_ab == RB_F16 || a->dtype_ab == RB_BF16 || a->dtype_ab == RB_F16S, "gemm_tc: operands must be fp16/bf16/split-fp16 (got %d)", a->dtype_ab);
    RB_REQUIRE(a->M > 0 && a->N > 0 && a->K > 0, "gemm_tc: empty problem");
    const bool split = a->dtype_ab == RB_F16S;
    RB_REQUIRE(!split || (a->A_lo && a->B_lo), "gemm_tc: split-fp16 operands need A_lo and B_lo");
    RB_REQUIRE(a->dtype_c != RB_F16S || a->C_lo, "gemm_tc: split-fp16 output needs C_lo");
    TcParams p;
    g_max_ctas = a->max_ctas;
    p.M = a->M; p.N = a->N; p.K = a->K;
    p.batch1 = a->batch1 > 0 ? a->batch1 : 1;
    const int batch0 = a->batch0 > 0 ? a->batch0 : 1;
    p.ntaps = a->ntaps > 1 ? a->ntaps : 1;
    p.k_per_tap = a->K / p.ntaps;
    for (int i = 0; i < 9; ++i) p.tap_rows[i] = a->tap_rows[i];
    p.trans_b = a->trans_b; p.is_bf16 = a->dtype_ab == RB_BF16;
    p.sc0 = a->sc0; p.sc1 = a->sc1; p.sr0 = a->sr0; p.sr1 = a->sr1; p.sna0 = a->sna0; p.snb0 = a->snb0;
    p.epi = make_epilogue(a);
    // A (M x K) at least as large as B (N x K): walk row bands, so that A streams from HBM once (refiner pointwise convolutions: up to
    // 93312 x 569 against 569 x 569); otherwise N-major, which re-reads the smaller A
    p.band_major = a->M >= a->N;
    p.clk = tc_clk_buffer();
    { static const int em = [] { const char* e = getenv("ROMAB200_GEMM_EPI"); return e && atoi(e) == 0 ? 0 : 2; }(); p.epi_mode = em; }
    if (p.ntaps > 1) {
        RB_REQUIRE(a->K % p.ntaps == 0 && p.k_per_tap % TC_BK == 0, "gemm_tc: K/ntaps=%d must be a multiple of %d", p.k_per_tap, TC_BK);
        RB_REQUIRE(!a->trans_b && batch0 * p.batch1 == 1, "gemm_tc: taps need un-batched [N,K] weights");
    }
    const int zdim = batch0 * p.batch1;
    RB_REQUIRE(zdim <= 65535, "gemm_tc: batch too large");
    const int64_t a_rows = a->a_rows > 0 ? a->a_rows : a->M;
    int BN = a->N <= 32 && !a->trans_b ? 32 : (a->N <= 64 ? 64 : (a->N <= 128 || a->trans_b ? 128 : 256));
    if (!a->trans_b && a->N > 128) {
        // UMMA N may be any multiple of 16: pick the tile width that wastes the fewest columns (C = 144 / 569 / 1137 ...)
        if (a->N <= 144) BN = 144;
        else if (a->N <= 192) BN = 192;
        else {
            const int w192 = (a->N + 191) / 192 * 192 - a->N, w256 = (a->N + 255) / 256 * 256 - a->N;
            BN = (w192 + a->N / 20 < w256) ? 192 : 256;
        }
    }
    // few tiles: keep 128-wide tiles so that more CTAs are in flight
    // (the threshold is in tiles: below ~100 wide tiles less than 2/3 of the SMs would have work; above it the wider tile wins
    // because these shapes are bound by L2 -> shared-memory operand traffic, which a 128-wide tile raises by a third)
    if (BN > 128 && ((int64_t)((a->M + 127) / 128) * ((a->N + BN - 1) / BN) * zdim) < 100) BN = 128;
    // CTA-pair candidates: all tiles of a launch take the same time, so the launch costs ceil(tiles / SM pairs) waves of a tile whose time
    // grows with BN.  When the 256-wide choice ends in a mostly empty last wave, 192-wide tiles finish earlier (ViT qkv, 3202 x 3072:
    // 156 tiles = 3 waves of 256 columns against 208 tiles = 3 waves of 192); a 5 % handicap keeps the wider tile on ties.  (Split ViT
    // fc1, 3202 x 4096, ties at 4 waves of 192 against 3 of 256: 192 with early release is faster alone, 86 against 93 us, but slower
    // inside the step, 2.29 against 2.13 ms, where it shares the GPU with the CNN branch; so the tie stays with 256.)
    if (!a->trans_b && BN == 256 && pair_mode() && wave_rule()) {
        const long long mt = (long long)((a->M + 255) / 256) * zdim, units = sm_count() / 2 > 0 ? sm_count() / 2 : 1;
        auto cost = [&](int bn) { const long long t = mt * ((a->N + bn - 1) / bn); return (t + units - 1) / units * bn; };
        if (mt * ((a->N + 255) / 256) >= 40 && cost(192) * 21 < cost(256) * 20) BN = 192;
    }
    {   // experiments: ROMAB200_GEMM_BN forces the tile width of the [N,K] layouts when it is one of the instantiated widths
        static const int force_bn = [] { const char* e = getenv("ROMAB200_GEMM_BN"); return e ? atoi(e) : 0; }();
        if (force_bn && !a->trans_b && (force_bn == 32 || force_bn == 64 || force_bn == 128 || force_bn == 144 || force_bn == 192 || force_bn == 256)) BN = force_bn;
    }
    // CTA-pair tiles (256 x BN, tcgen05 cta_group::2): half the B-operand traffic per MMA; for the [N,K] layouts with enough
    // 256-row tiles to fill the 74 SM pairs
    int pair_bn = 0;
    if (!a->trans_b && pair_mode() && (BN == 256 || BN == 192)) {
        const long long pair_tiles = (long long)((a->M + 255) / 256) * ((a->N + BN - 1) / BN) * zdim;
        if (pair_mode() == 2 || pair_tiles >= 40) pair_bn = BN;
        // split operands: a 256-wide tile's two accumulators fill TMEM, so its drain is exposed; 128-wide pair tiles double-buffer them
        static const int split_pair_bn = [] { const char* e = getenv("ROMAB200_GEMM_SPLIT_PAIR_BN"); return e ? atoi(e) : 0; }();
        if (pair_bn && split && split_pair_bn == 128 && a->N % 128 == 0) pair_bn = 128;
    }
    TcMaps maps;
    const uint64_t a_inner = p.ntaps > 1 ? p.k_per_tap : a->K;
    if (make_map(&maps.a, a->A, p.is_bf16, a_inner, a_rows, a->lda, p.batch1, a->sa1, batch0, a->sa0, TC_BK, TC_BM)) return 1;
    if (split && make_map(&maps.a_lo, a->A_lo, 0, a_inner, a_rows, a->lda, p.batch1, a->sa1, batch0, a->sa0, TC_BK, TC_BM)) return 1;
    if (!a->trans_b) {
        const uint32_t box_n = pair_bn ? pair_bn / 2 : BN;      // a CTA of a pair loads its half of the B tile
        if (make_map(&maps.b, a->B, p.is_bf16, a->K, a->N, a->ldb, p.batch1, a->sb1, batch0, a->sb0, TC_BK, box_n)) return 1;
        if (split && make_map(&maps.b_lo, a->B_lo, 0, a->K, a->N, a->ldb, p.batch1, a->sb1, batch0, a->sb0, TC_BK, box_n)) return 1;
    } else {
        if (make_map(&maps.b, a->B, p.is_bf16, a->N, a->K, a->ldb, p.batch1, a->sb1, batch0, a->sb0, 64, TC_BK)) return 1;
        if (split && make_map(&maps.b_lo, a->B_lo, 0, a->N, a->K, a->ldb, p.batch1, a->sb1, batch0, a->sb0, 64, TC_BK)) return 1;
    }
    if (!split) { maps.a_lo = maps.a; maps.b_lo = maps.b; }
    // TMA-store epilogue when the output is a plain (or zero-bordered) matrix with 16-byte aligned pitches; an in-place fp32 residual
    // (R == C: the residual stream, the GP trailing update) becomes a reduce-add.  Otherwise the per-lane direct stores.
    maps.c = maps.a; maps.c_lo = maps.a;
    {
        const int es_c = a->dtype_c == RB_F32 ? 4 : 2;
        const bool align_ok = ((uintptr_t)a->C) % 16 == 0 && (a->ldc * es_c) % 16 == 0 && (p.batch1 <= 1 || (a->sc1 * es_c) % 16 == 0) &&
                              (batch0 <= 1 || (a->sc0 * es_c) % 16 == 0) && (a->dtype_c != RB_F16S || ((uintptr_t)a->C_lo) % 16 == 0);
        const bool rowmap_ok = a->rowmap == RB_ROWMAP_NONE || a->rowmap == RB_ROWMAP_PAD_KEEP;
        const bool inplace_r = a->R && a->R == a->C && a->dtype_r == RB_F32 && a->dtype_c == RB_F32 && a->ldr == a->ldc && a->sr0 == a->sc0 && a->sr1 == a->sc1 &&
                               a->epi == RB_EPI_LINEAR;
        if (p.epi_mode >= 2 && align_ok && rowmap_ok && (!a->R || inplace_r)) {
            const uint32_t box_cols = (a->dtype_c == RB_F16 || a->dtype_c == RB_BF16) ? 32 : 16;
            const int dt = a->dtype_c == RB_F16S ? RB_F16 : a->dtype_c;
            if (make_out_map(&maps.c, a->C, dt, a->N, a->M, a->ldc, p.batch1, a->sc1, batch0, a->sc0, box_cols)) return 1;
            if (a->dtype_c == RB_F16S && make_out_map(&maps.c_lo, a->C_lo, RB_F16, a->N, a->M, a->ldc, p.batch1, a->sc1, batch0, a->sc0, box_cols)) return 1;
            p.epi_mode = inplace_r ? 3 : 2;
            if (inplace_r) p.epi.R = nullptr;           // the reduction adds it
        } else if (p.epi_mode >= 2) {
            p.epi_mode = 0;
        }
    }
    if (pair_bn == 128) return launch_tc_pair<128, true>(maps, p, zdim, stream);
    if (pair_bn == 256) return split ? launch_tc_pair<256, true>(maps, p, zdim, stream) : launch_tc_pair<256, false>(maps, p, zdim, stream);
    if (pair_bn == 192) return split ? launch_tc_pair<192, true>(maps, p, zdim, stream) : launch_tc_pair<192, false>(maps, p, zdim, stream);
    return split ? dispatch_tc<true>(BN, maps, p, zdim, stream) : dispatch_tc<false>(BN, maps, p, zdim, stream);
}

}  // namespace rb

// debug: read (and optionally reset) the role-time counters collected with ROMAB200_TC_CLK=1 (16 x u64, see gemm_tc.cu)
extern "C" int romab200_debug_tc_clk(unsigned long long* out, int reset) {
    unsigned long long* buf = rb::tc_clk_buffer();
    if (!buf) return 1;
    if (cudaMemcpy(out, buf, 16 * sizeof(unsigned long long), cudaMemcpyDeviceToHost) != cudaSuccess) return 2;
    if (reset) cudaMemset(buf, 0, 16 * sizeof(unsigned long long));
    return 0;
}
