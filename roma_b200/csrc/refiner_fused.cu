// Fused ConvRefiner block for the stride-2 maps (C = 144):  out = PW_{144x144}( ReLU( BN( DW5x5(in) ) ) ) + bias
// (create_block, romatch/models/matcher.py:92-122) in ONE kernel: the activation map is read once and written once.
// Un-fused, this block is a depthwise kernel plus a GEMM that together move the 107 MB map four times and spend most
// of their time in per-tile overheads; here
//   * 1 thread TMA-loads the 12x20 pixel input window of an 8x16 tile (4-D tensor map over [B,H,W,C]: the image border
//     is the map's out-of-bounds zero fill, no address arithmetic, no registers);
//   * 9 depthwise warps run the 5x5 stage on the CUDA cores (channel pairs, packed FFMA2) and write the ReLU'd
//     128 x 144 result straight into the 128B-swizzled K-major layout of a UMMA A operand;
//   * 1 thread issues 9 tcgen05.mma (M=128, N=144, K=16) against the pointwise weights, which were TMA-loaded into
//     shared memory once and stay resident;
//   * 4 epilogue warps read the fp32 accumulator from TMEM (double-buffered), add the bias and store 16-bit rows.
// refiner_block_c144_split_kernel (below) is the same block on fp32 maps with split-fp16 pointwise operands (parity mode),
// bit-identical to the depthwise kernel + split GEMM pair it replaces.
#include "common.cuh"
#include <cuda.h>

namespace rb {
namespace fz {
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
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
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
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
// UMMA shared-memory descriptor; layout 2 = SWIZZLE_128B, 4 = SWIZZLE_64B
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout = 2) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)layout << 61;
    return d;
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
}  // namespace fz

#ifdef RB_FZ_CLK
__device__ long long g_fz_clk[64];
#define FZCLK(var) const long long var = clock64();
#else
#define FZCLK(var)
#endif

struct FusedParams {
    const void* in; void* out; int64_t ld;
    const float* dw_w; int64_t ldw; const float* dw_b; const float* pw_b;
    int batch, H, W, tiles_x, tiles_y, total_tiles, is_bf16;
};

constexpr int FZ_C = 144, FZ_CP = 72, FZ_TH = 8, FZ_TW = 16, FZ_IH = 12, FZ_IW = 20;
constexpr int FZ_DW_THREADS = 288;                    // 72 channel pairs x 4 row groups
constexpr int FZ_THREADS = 32 + 128 + FZ_DW_THREADS + 32;  // warp 0: weights + MMA, warps 1-4: epilogue, warps 5-13: depthwise, warp 14: input TMA
constexpr int FZ_IN_BYTES = FZ_IH * FZ_IW * FZ_C * 2;              // 69120
constexpr int FZ_A_BYTES = 3 * 128 * 128;                          // 49152: 3 k-blocks of 64 channels, 128 pixel rows
constexpr int FZ_B_KB = FZ_C * 128;                                // 18432 per k-block
constexpr int FZ_B_BYTES = 3 * FZ_B_KB;                            // 55296
constexpr int FZ_W_BYTES = 25 * FZ_C * 4;                          // depthwise taps, fp32, tap-major
constexpr int FZ_SMEM = FZ_A_BYTES + FZ_B_BYTES + FZ_IN_BYTES + FZ_W_BYTES + 1024 + 1024;

template <typename T>
__global__ void __launch_bounds__(FZ_THREADS, 1) refiner_block_c144_kernel(const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_in, const FusedParams p) {
    rb::pdl_wait();
    using namespace fz;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - ((uint32_t)__cvta_generic_to_shared(smem_raw) & 1023u)) & 1023u);   // offset on the array: keeps ld/st.shared
    uint8_t* sA = smem;
    uint8_t* sB = sA + FZ_A_BYTES;
    uint8_t* sIn = sB + FZ_B_BYTES;
    float* s_dw = reinterpret_cast<float*>(sIn + FZ_IN_BYTES);            // [25][144]
    uint64_t* bars = reinterpret_cast<uint64_t*>(sIn + FZ_IN_BYTES + FZ_W_BYTES);
    uint64_t* w_full = bars;            // weights landed
    uint64_t* a_full = bars + 1;        // depthwise tile written (9 warp arrivals)
    uint64_t* a_empty = bars + 2;       // MMAs that read it retired
    uint64_t* t_full = bars + 3;        // [2] accumulator ready
    uint64_t* t_empty = bars + 5;       // [2] accumulator drained (4 warp arrivals)
    uint64_t* in_full = bars + 7;       // input window landed (TMA transaction bytes)
    uint64_t* in_empty = bars + 8;      // depthwise warps have read it (9 warp arrivals)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);
    float* s_bias = reinterpret_cast<float*>(bars + 10);    // [144]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        mbar_init(w_full, 1); mbar_init(a_full, FZ_DW_THREADS / 32); mbar_init(a_empty, 1);
        for (int s = 0; s < 2; ++s) { mbar_init(&t_full[s], 1); mbar_init(&t_empty[s], 4); }
        mbar_init(in_full, 1); mbar_init(in_empty, FZ_DW_THREADS / 32);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(tmem_slot, 512);
    for (int i = threadIdx.x; i < FZ_C; i += FZ_THREADS) s_bias[i] = p.pw_b[i];
    for (int i = threadIdx.x; i < 25 * FZ_C; i += FZ_THREADS) s_dw[i] = p.dw_w[(int64_t)(i / FZ_C) * p.ldw + (i % FZ_C)];
    for (int i = threadIdx.x; i < FZ_A_BYTES / 16; i += FZ_THREADS) reinterpret_cast<uint4*>(sA)[i] = make_uint4(0u, 0u, 0u, 0u);   // K padding stays 0
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int tiles_per_img = p.tiles_x * p.tiles_y;

    if (warp == 0) {
        if (lane == 0) {
            // pointwise weights [144 x 144] -> three K-major k-blocks, loaded once for the whole persistent kernel
            mbar_expect_tx(w_full, FZ_B_BYTES);
            for (int kb = 0; kb < 3; ++kb) tma_load_2d(sB + kb * FZ_B_KB, &map_w, w_full, kb * 64, 0);
            const uint32_t fmt = p.is_bf16 ? 1u : 0u;
            const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(FZ_C >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
            mbar_wait(w_full, 0);
            const uint32_t a_addr = smem_u32(sA), b_addr = smem_u32(sB);
            uint32_t it = 0;
            for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
                const uint32_t acc = it & 1;
                mbar_wait(&t_empty[acc], ((it >> 1) & 1) ^ 1);
                mbar_wait(a_full, it & 1);
                tc_fence_after();
#pragma unroll
                for (int k = 0; k < FZ_C / 16; ++k) {
                    const uint32_t aoff = (k >> 2) * (128 * 128) + (k & 3) * 32, boff = (k >> 2) * FZ_B_KB + (k & 3) * 32;
                    umma_f16(tmem_base + acc * FZ_C, smem_desc(a_addr + aoff, 16, 1024), smem_desc(b_addr + boff, 16, 1024), idesc, k != 0);
                }
                umma_commit(a_empty);
                umma_commit(&t_full[acc]);
            }
        }
    } else if (warp <= 4) {
        // ===== epilogue: TMEM -> + bias -> 16-bit rows (one pixel per thread, 288 contiguous bytes) =====
        const int q = warp & 3;
        const int m = q * 32 + lane;                       // pixel of the tile
        const int py = m / FZ_TW, px = m - py * FZ_TW;
        uint32_t it = 0;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
            const int img = tile / tiles_per_img, r = tile - img * tiles_per_img;
            const int ty = r / p.tiles_x, tx = r - ty * p.tiles_x;
            const int yy = ty * FZ_TH + py, xx = tx * FZ_TW + px;
            const bool live = yy < p.H && xx < p.W;
            T* orow = (T*)p.out + (((int64_t)img * p.H + yy) * p.W + xx) * p.ld;
            const uint32_t acc = it & 1;
            mbar_wait(&t_full[acc], (it >> 1) & 1);
            tc_fence_after();
#pragma unroll 1
            for (int cb = 0; cb < FZ_C; cb += 32) {
                float v[32];
                tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + acc * FZ_C + cb, v);
                if (!live) continue;
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    if (cb + 8 * g < FZ_C) {
                        T pk[8];
#pragma unroll
                        for (int e = 0; e < 8; ++e) pk[e] = from_f<T>(v[8 * g + e] + s_bias[cb + 8 * g + e]);
                        *reinterpret_cast<uint4*>(orow + cb + 8 * g) = *reinterpret_cast<uint4*>(pk);
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&t_empty[acc]);
        }
    } else if (warp == 14) {
        // ===== input loader: one TMA box per tile, re-armed as soon as the depthwise warps have read the previous window =====
        if (lane == 0) {
            uint32_t it = 0;
            for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
                const int img = tile / tiles_per_img, r = tile - img * tiles_per_img;
                const int ty = r / p.tiles_x, tx = r - ty * p.tiles_x;
                if (it > 0) mbar_wait(in_empty, (it - 1) & 1);
                mbar_expect_tx(in_full, FZ_IN_BYTES);
                tma_load_4d(sIn, &map_in, in_full, 0, tx * FZ_TW - 2, ty * FZ_TH - 2, img);
            }
        }
    } else {
        // ===== depthwise producers: thread = (channel pair, 2 output rows) =====
        const int t = threadIdx.x - 160;                   // 0 .. 287
        const int cp = t % FZ_CP, rg = t / FZ_CP;
        const float2 bv = make_float2(p.dw_b[2 * cp], p.dw_b[2 * cp + 1]);
        // A-operand address pieces of this thread's two channels (K-major, 128B swizzle): k-block, 16-byte chunk, byte in chunk
        const int kb = cp >> 5, chunk = (cp & 31) >> 2, inb = (cp & 3) * 4;
        uint32_t it = 0;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
            FZCLK(t0)
            mbar_wait(in_full, it & 1);
            FZCLK(t1)
            // filter taps: re-read from shared memory per tile so that they are not live during the load phase
            float2 wv[25];
#pragma unroll
            for (int k = 0; k < 25; ++k) wv[k] = *reinterpret_cast<const float2*>(&s_dw[k * FZ_C + 2 * cp]);
            float2 acc2[2][FZ_TW];
#pragma unroll
            for (int rr = 0; rr < 2; ++rr)
#pragma unroll
                for (int i = 0; i < FZ_TW; ++i) acc2[rr][i] = bv;
#pragma unroll
            for (int iy = 0; iy < 6; ++iy) {
#pragma unroll
                for (int ix = 0; ix < FZ_IW; ++ix) {
                    T pr[2];
                    *reinterpret_cast<uint32_t*>(pr) = *reinterpret_cast<const uint32_t*>(sIn + ((2 * rg + iy) * FZ_IW + ix) * (FZ_C * 2) + cp * 4);
                    const float2 v = make_float2(to_f(pr[0]), to_f(pr[1]));
#pragma unroll
                    for (int rr = 0; rr < 2; ++rr) {
                        const int ky = iy - rr;
                        if (ky >= 0 && ky < 5) {
#pragma unroll
                            for (int kx = 0; kx < 5; ++kx) {
                                const int ox = ix - kx;
                                if (ox >= 0 && ox < FZ_TW) acc2[rr][ox] = __ffma2_rn(wv[ky * 5 + kx], v, acc2[rr][ox]);
                            }
                        }
                    }
                }
            }
            FZCLK(t2)
            __syncwarp();
            if (lane == 0) mbar_arrive(in_empty);          // this warp's reads of the input window are done
            mbar_wait(a_empty, (it & 1) ^ 1);
            FZCLK(t3)              // the MMAs of the previous tile no longer read sA
#pragma unroll
            for (int rr = 0; rr < 2; ++rr) {
#pragma unroll
                for (int i = 0; i < FZ_TW; ++i) {
                    const int m = (2 * rg + rr) * FZ_TW + i;
                    T pair[2] = {from_f<T>(fmaxf(acc2[rr][i].x, 0.f)), from_f<T>(fmaxf(acc2[rr][i].y, 0.f))};
                    *reinterpret_cast<uint32_t*>(sA + kb * (128 * 128) + m * 128 + ((chunk ^ (m & 7)) << 4) + inb) = *reinterpret_cast<uint32_t*>(pair);
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(a_full);
#ifdef RB_FZ_CLK
            if (blockIdx.x == 0 && lane == 0) { const long long t4 = clock64(); long long* g = g_fz_clk + (warp - 5) * 5; g[0] += t1 - t0; g[1] += t2 - t1; g[2] += t3 - t2; g[3] += t4 - t3; g[4] += 1; }
#endif
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) { tc_fence_after(); tmem_dealloc(tmem_base, 512); }
}

// ---------------------------------------------------------------------------------------------------------------------
// The same block on fp32 maps (parity mode), with the pointwise GEMM on split-fp16 operand pairs: one kernel in place of
// dwconv5x5_relu_tma_kernel<float> (fp32 map -> RB_F16S pair in memory) followed by gemm_tc_kernel<144, SPLIT>.  Both
// halves do exactly the arithmetic of those two kernels, so the output is bit-identical to theirs:
//   * depthwise: accumulator = bias, 25 packed FFMA2 per output in (ky, kx) order, ReLU, hi = fp16(x), lo = fp16((x - hi) * 2^11);
//   * pointwise: per k-step of 16, acc0 += A_hi.B_hi, then acc1 += A_hi.B_lo and acc1 += A_lo.B_hi, k ascending (9 steps);
//   * epilogue: acc0 + acc1 * 2^-11 (one fmaf), then + bias, stored as fp32.
// The fp32 window of all 144 channels (138 KB) does not fit beside the resident weights, so a tile is streamed in five
// 32-channel chunks (the last 16 wide: its upper half is the tensor map's zero fill and is never read by an MMA):
//   * warp 5, one thread: TMA-loads the 12 x 20 pixel x 32 channel fp32 window of a chunk into a 3-stage ring;
//   * warps 6-13 (256 threads = 16 channel pairs x 4 row pairs x 4 column quarters, 2 x 4 outputs each) run the depthwise
//     stage of the chunk and write its hi / lo planes into a 64B-swizzled K-major A stage (two stages);
//   * warp 0, one thread: issues the 2 (last chunk: 1) k-steps of the chunk as soon as its A stage is written;
//   * warps 1-4: drain the two accumulators (288 of 512 TMEM columns: single-buffered), release TMEM after the last load, and
//     store fp32 rows through TMA (16 channels x 16 pixels x 2 rows per store; image borders clipped by the tensor map).
//     This overlaps the depthwise stage of the first chunks of the next tile.
// Shared memory (bytes): B hi + lo, 5 chunks x 144 rows x 64 B each   92160
//                        A hi + lo, 2 stages x 128 rows x 64 B each   32768
//                        input windows, 3 x 12 x 20 x 32 x 4          92160
//                        epilogue staging, 4 warps x 2 KB              8192
//                        bias, barriers, TMEM slot, 1 KB alignment     1792   -> 227072 of 232448, one CTA per SM
// The depthwise taps (14 KB) are read per chunk from global memory through L1; there is no room for them here.
constexpr int FS_CH = 32, FS_NCHUNK = 5, FS_WIN_STAGES = 2 + 1;
constexpr int FS_DW_THREADS = 256;
constexpr int FS_THREADS = 32 + 128 + 32 + FS_DW_THREADS;   // warp 0: weights + MMA, warps 1-4: epilogue, warp 5: input TMA, warps 6-13: depthwise
constexpr int FS_WIN_BYTES = FZ_IH * FZ_IW * FS_CH * 4;     // 30720
constexpr int FS_B_CHUNK = FZ_C * FS_CH * 2;                // 9216: 144 rows x 64 B
constexpr int FS_B_PLANE = FS_NCHUNK * FS_B_CHUNK;          // 46080
constexpr int FS_A_PLANE = 128 * FS_CH * 2;                 // 8192
constexpr int FS_A_STAGE = 2 * FS_A_PLANE;                  // hi + lo
constexpr int FS_OUT_WARP = 32 * 16 * 4;                    // 2048: 32 pixels x 16 fp32 channels
constexpr int FS_OFF_A = 2 * FS_B_PLANE;
constexpr int FS_OFF_WIN = FS_OFF_A + 2 * FS_A_STAGE;
constexpr int FS_OFF_OUT = FS_OFF_WIN + FS_WIN_STAGES * FS_WIN_BYTES;
constexpr int FS_OFF_BIAS = FS_OFF_OUT + 4 * FS_OUT_WARP;
constexpr int FS_OFF_BAR = FS_OFF_BIAS + FS_NCHUNK * FS_CH * 4;
constexpr int FS_SMEM = FS_OFF_BAR + 128 + 1024;
static_assert(FS_SMEM <= 232448, "shared memory budget");

struct FusedSplitParams {
    const float* dw_w; int64_t ldw; const float* dw_b; const float* pw_b;
    int H, W, tiles_x, tiles_y, total_tiles;
};

__global__ void __launch_bounds__(FS_THREADS, 1)
refiner_block_c144_split_kernel(const __grid_constant__ CUtensorMap map_w_hi, const __grid_constant__ CUtensorMap map_w_lo,
                                const __grid_constant__ CUtensorMap map_in, const __grid_constant__ CUtensorMap map_out, const FusedSplitParams p) {
    rb::pdl_wait();
    using namespace fz;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - ((uint32_t)__cvta_generic_to_shared(smem_raw) & 1023u)) & 1023u);
    uint8_t* sB = smem;                                   // [hi | lo][chunk][144 rows][64 B], 64B-swizzled
    uint8_t* sA = smem + FS_OFF_A;                        // [stage][hi | lo][128 rows][64 B], 64B-swizzled
    uint8_t* sWin = smem + FS_OFF_WIN;                    // [stage][12 rows][20 pixels][32 channels] fp32
    uint8_t* sOut = smem + FS_OFF_OUT;                    // [epilogue warp][32 pixels][16 channels] fp32
    float* s_bias = reinterpret_cast<float*>(smem + FS_OFF_BIAS);   // [160], zero beyond 144
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + FS_OFF_BAR);
    uint64_t* w_full = bars;              // pointwise weights landed
    uint64_t* win_full = bars + 1;        // [3] input window landed (TMA transaction bytes)
    uint64_t* win_empty = bars + 4;       // [3] depthwise warps have read it (8 warp arrivals)
    uint64_t* a_full = bars + 7;          // [2] A stage written (8 warp arrivals)
    uint64_t* a_empty = bars + 9;         // [2] MMAs that read it retired
    uint64_t* t_full = bars + 11;         // accumulators complete
    uint64_t* t_empty = bars + 12;        // accumulators drained (4 warp arrivals)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 13);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        mbar_init(w_full, 1);
        for (int s = 0; s < FS_WIN_STAGES; ++s) { mbar_init(&win_full[s], 1); mbar_init(&win_empty[s], FS_DW_THREADS / 32); }
        for (int s = 0; s < 2; ++s) { mbar_init(&a_full[s], FS_DW_THREADS / 32); mbar_init(&a_empty[s], 1); }
        mbar_init(t_full, 1); mbar_init(t_empty, 4);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(tmem_slot, 512);
    for (int i = threadIdx.x; i < FS_NCHUNK * FS_CH; i += FS_THREADS) s_bias[i] = i < FZ_C ? p.pw_b[i] : 0.f;
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int tiles_per_img = p.tiles_x * p.tiles_y;

    if (warp == 0) {
        if (lane == 0) {
            // pointwise weights: both planes as five 32-wide k-chunks, loaded once for the whole persistent kernel
            mbar_expect_tx(w_full, 2 * FS_B_PLANE);
            for (int c = 0; c < FS_NCHUNK; ++c) {
                tma_load_2d(sB + c * FS_B_CHUNK, &map_w_hi, w_full, c * FS_CH, 0);
                tma_load_2d(sB + FS_B_PLANE + c * FS_B_CHUNK, &map_w_lo, w_full, c * FS_CH, 0);
            }
            const uint32_t idesc = (1u << 4) | ((uint32_t)(FZ_C >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);   // f32 += f16 x f16, K-major
            mbar_wait(w_full, 0);
            const uint32_t a_addr = smem_u32(sA), b_addr = smem_u32(sB);
            uint32_t it = 0, j = 0;
            for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
                mbar_wait(t_empty, (it & 1) ^ 1);
                tc_fence_after();
#pragma unroll
                for (int c = 0; c < FS_NCHUNK; ++c, ++j) {
                    const uint32_t s = j & 1;
                    mbar_wait(&a_full[s], (j >> 1) & 1);
                    tc_fence_after();
                    const uint32_t a_hi = a_addr + s * FS_A_STAGE, a_lo = a_hi + FS_A_PLANE;
                    const uint32_t b_hi = b_addr + c * FS_B_CHUNK, b_lo = b_hi + FS_B_PLANE;
#pragma unroll
                    for (int ks = 0; ks < 2; ++ks) {
                        if (2 * c + ks < FZ_C / 16) {          // k-steps beyond K = 144 are skipped, as in gemm_tc
                            const uint32_t accum = (c | ks) != 0;
                            const uint64_t dah = smem_desc(a_hi + 32 * ks, 16, 512, 4), dal = smem_desc(a_lo + 32 * ks, 16, 512, 4);
                            const uint64_t dbh = smem_desc(b_hi + 32 * ks, 16, 512, 4), dbl = smem_desc(b_lo + 32 * ks, 16, 512, 4);
                            umma_f16(tmem_base, dah, dbh, idesc, accum);
                            umma_f16(tmem_base + FZ_C, dah, dbl, idesc, accum);
                            umma_f16(tmem_base + FZ_C, dal, dbh, idesc, 1u);
                        }
                    }
                    umma_commit(&a_empty[s]);
                }
                umma_commit(t_full);
            }
        }
    } else if (warp <= 4) {
        // ===== epilogue: TMEM -> acc0 + acc1 * 2^-11 + bias -> fp32 rows through TMA stores =====
        const int q = warp & 3;                            // TMEM lane quarter = pixels 32q .. 32q + 31 = tile rows 2q, 2q + 1
        uint8_t* stage = sOut + (warp - 1) * FS_OUT_WARP;
        uint32_t it = 0;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
            const int img = tile / tiles_per_img, r = tile - img * tiles_per_img;
            const int ty = r / p.tiles_x, tx = r - ty * p.tiles_x;
            const int y0 = ty * FZ_TH + 2 * q;
            mbar_wait(t_full, it & 1);
            tc_fence_after();
#pragma unroll 1
            for (int cb = 0; cb < FZ_C; cb += 32) {
                float v[32], w[32];
                tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + cb, v);
                tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + FZ_C + cb, w);
                if (cb + 32 >= FZ_C) {                         // last chunk read: the MMA thread may start the next tile
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(t_empty);
                }
#pragma unroll
                for (int k = 0; k < 32; ++k) v[k] = fmaf(w[k], 1.0f / 2048.0f, v[k]);
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const float4 b4 = *reinterpret_cast<const float4*>(&s_bias[cb + 4 * k]);
                    v[4 * k] += b4.x; v[4 * k + 1] += b4.y; v[4 * k + 2] += b4.z; v[4 * k + 3] += b4.w;
                }
                if (y0 >= p.H) continue;                       // warp-uniform: both rows below the image
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    if (cb + 16 * h >= FZ_C) break;
                    if (lane == 0) bulk_wait_read();           // the previous store has read the staging buffer
                    __syncwarp();
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        *reinterpret_cast<float4*>(stage + lane * 64 + 16 * k) = make_float4(v[16 * h + 4 * k], v[16 * h + 4 * k + 1], v[16 * h + 4 * k + 2], v[16 * h + 4 * k + 3]);
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) { tma_store_4d(&map_out, stage, cb + 16 * h, tx * FZ_TW, y0, img); bulk_commit(); }
                }
            }
        }
        if (lane == 0) bulk_wait_all();
        __syncwarp();
    } else if (warp == 5) {
        // ===== input loader: one TMA box per (tile, chunk), 3 windows in flight =====
        if (lane == 0) {
            uint32_t j = 0;
            for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
                const int img = tile / tiles_per_img, r = tile - img * tiles_per_img;
                const int ty = r / p.tiles_x, tx = r - ty * p.tiles_x;
                for (int c = 0; c < FS_NCHUNK; ++c, ++j) {
                    const uint32_t s = j % FS_WIN_STAGES;
                    if (j >= FS_WIN_STAGES) mbar_wait(&win_empty[s], (j / FS_WIN_STAGES - 1) & 1);
                    mbar_expect_tx(&win_full[s], FS_WIN_BYTES);
                    tma_load_4d(sWin + s * FS_WIN_BYTES, &map_in, &win_full[s], c * FS_CH, tx * FZ_TW - 2, ty * FZ_TH - 2, img);
                }
            }
        }
    } else {
        // ===== depthwise: thread = (channel pair, 2 output rows, 4 output columns) of the chunk =====
        const int t = threadIdx.x - 192;                   // 0 .. 255
        const int pr = t & 15, xq = (t >> 4) & 3, rg = t >> 6;
        const int sw_chunk = pr >> 2, inb = (pr & 3) * 4;  // 16-byte chunk and byte of this pair in a 64-byte A row
        uint32_t j = 0;
        for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
#pragma unroll 1
            for (int c = 0; c < FS_NCHUNK; ++c, ++j) {
                const int ch = c * FS_CH + 2 * pr;
                const bool ok = ch < FZ_C;                 // the upper half of the last chunk computes zeros that no MMA reads
                float2 wv[25];
#pragma unroll
                for (int k = 0; k < 25; ++k) wv[k] = ok ? __ldg(reinterpret_cast<const float2*>(p.dw_w + k * p.ldw + ch)) : make_float2(0.f, 0.f);
                const float2 bv = ok ? __ldg(reinterpret_cast<const float2*>(p.dw_b + ch)) : make_float2(0.f, 0.f);
                const uint32_t s = j % FS_WIN_STAGES;
                mbar_wait(&win_full[s], (j / FS_WIN_STAGES) & 1);
                const float* win = reinterpret_cast<const float*>(sWin + s * FS_WIN_BYTES);
                float2 acc[2][4];
#pragma unroll
                for (int rr = 0; rr < 2; ++rr)
#pragma unroll
                    for (int i = 0; i < 4; ++i) acc[rr][i] = bv;
#pragma unroll
                for (int iy = 0; iy < 6; ++iy) {
#pragma unroll
                    for (int ix = 0; ix < 8; ++ix) {
                        const float2 v = *reinterpret_cast<const float2*>(&win[((2 * rg + iy) * FZ_IW + 4 * xq + ix) * FS_CH + 2 * pr]);
#pragma unroll
                        for (int rr = 0; rr < 2; ++rr) {
                            const int ky = iy - rr;
                            if (ky >= 0 && ky < 5) {
#pragma unroll
                                for (int kx = 0; kx < 5; ++kx) {
                                    const int ox = ix - kx;
                                    if (ox >= 0 && ox < 4) acc[rr][ox] = __ffma2_rn(wv[ky * 5 + kx], v, acc[rr][ox]);
                                }
                            }
                        }
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&win_empty[s]);
                const uint32_t as = j & 1;
                mbar_wait(&a_empty[as], ((j >> 1) & 1) ^ 1);   // the MMAs of chunk j - 2 no longer read this A stage
                uint8_t* a_hi = sA + as * FS_A_STAGE;
#pragma unroll
                for (int rr = 0; rr < 2; ++rr) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int m = (2 * rg + rr) * FZ_TW + 4 * xq + i;
                        __half hi[2], lo[2];
                        split_f16s(fmaxf(acc[rr][i].x, 0.f), hi[0], lo[0]);
                        split_f16s(fmaxf(acc[rr][i].y, 0.f), hi[1], lo[1]);
                        const int off = m * 64 + ((sw_chunk ^ ((m >> 1) & 3)) << 4) + inb;
                        *reinterpret_cast<uint32_t*>(a_hi + off) = *reinterpret_cast<uint32_t*>(hi);
                        *reinterpret_cast<uint32_t*>(a_hi + FS_A_PLANE + off) = *reinterpret_cast<uint32_t*>(lo);
                    }
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(&a_full[as]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) { tc_fence_after(); tmem_dealloc(tmem_base, 512); }
}

typedef CUresult (*EncodeTiledFnFz)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
}  // namespace rb

using namespace rb;

#ifdef RB_FZ_CLK
extern "C" int romab200_debug_fzclk(long long* out, int reset) {
    if (reset) { long long z[64] = {0}; return (int)cudaMemcpyToSymbol(rb::g_fz_clk, z, sizeof(z)); }
    return (int)cudaMemcpyFromSymbol(out, rb::g_fz_clk, sizeof(long long) * 64);
}
#endif

// fp32 maps, split-fp16 pointwise weights (pw_weight = hi plane, pw_weight_lo = lo plane)
static int refiner_block_c144_split(const rb_refiner_block_c144_args* a, cudaStream_t st, EncodeTiledFnFz enc) {
    RB_REQUIRE(a->ld % 4 == 0 && a->ld >= FZ_C && ((uintptr_t)a->in) % 16 == 0 && ((uintptr_t)a->out) % 16 == 0 && a->in != a->out,
               "refiner_block_c144: bad fp32 activation layout");
    RB_REQUIRE(a->pw_weight_lo && ((uintptr_t)a->pw_weight_lo) % 16 == 0, "refiner_block_c144: fp32 maps need the lo plane of the split weights (pw_weight_lo)");
    RB_REQUIRE(a->ldw % 2 == 0 && ((uintptr_t)a->dw_weight) % 8 == 0 && ((uintptr_t)a->dw_bias) % 8 == 0, "refiner_block_c144: bad depthwise weight layout");
    CUtensorMap map_w[2];        // weight planes [144 x ld_pw] fp16: boxes of 32 (k) x 144 (n), 64B-swizzled K-major
    for (int i = 0; i < 2; ++i) {
        cuuint64_t dims[2] = {(cuuint64_t)FZ_C, (cuuint64_t)FZ_C};
        cuuint64_t strides[1] = {(cuuint64_t)a->ld_pw * 2};
        cuuint32_t box[2] = {(cuuint32_t)FS_CH, (cuuint32_t)FZ_C};
        cuuint32_t estr[2] = {1, 1};
        CUresult r = enc(&map_w[i], CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(i ? a->pw_weight_lo : a->pw_weight), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        RB_REQUIRE(r == CUDA_SUCCESS, "refiner_block_c144: cuTensorMapEncodeTiled (weights) failed with %d", (int)r);
    }
    // activations [B, H, W, 144] fp32 with pitch ld: input boxes 12 x 20 pixels x 32 channels (borders and the channel tail zero-filled),
    // output boxes 2 x 16 pixels x 16 channels (clipped at the borders)
    CUtensorMap map_in, map_out;
    cuuint64_t d4[4] = {(cuuint64_t)FZ_C, (cuuint64_t)a->w, (cuuint64_t)a->h, (cuuint64_t)a->batch};
    cuuint64_t s4[3] = {(cuuint64_t)a->ld * 4, (cuuint64_t)a->w * a->ld * 4, (cuuint64_t)a->h * a->w * a->ld * 4};
    cuuint32_t e4[4] = {1, 1, 1, 1};
    cuuint32_t bin[4] = {(cuuint32_t)FS_CH, (cuuint32_t)FZ_IW, (cuuint32_t)FZ_IH, 1};
    CUresult r = enc(&map_in, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<void*>(a->in), d4, s4, bin, e4, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    RB_REQUIRE(r == CUDA_SUCCESS, "refiner_block_c144: cuTensorMapEncodeTiled (input) failed with %d", (int)r);
    cuuint32_t bout[4] = {16, (cuuint32_t)FZ_TW, 2, 1};
    r = enc(&map_out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, a->out, d4, s4, bout, e4, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    RB_REQUIRE(r == CUDA_SUCCESS, "refiner_block_c144: cuTensorMapEncodeTiled (output) failed with %d", (int)r);
    FusedSplitParams p;
    p.dw_w = a->dw_weight; p.ldw = a->ldw; p.dw_b = a->dw_bias; p.pw_b = a->pw_bias;
    p.H = a->h; p.W = a->w; p.tiles_x = (a->w + FZ_TW - 1) / FZ_TW; p.tiles_y = (a->h + FZ_TH - 1) / FZ_TH;
    const long long total = (long long)p.tiles_x * p.tiles_y * a->batch;
    RB_REQUIRE(total > 0 && total < (1ll << 31), "refiner_block_c144: bad tile count");
    p.total_tiles = (int)total;
    const int dev = current_device();
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    static bool cfg[64] = {};            // function attributes are per device
    if (!cfg[dev & 63]) {
        RB_REQUIRE(cudaFuncSetAttribute(refiner_block_c144_split_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, FS_SMEM) == cudaSuccess, "refiner_block_c144: smem attribute");
        cfg[dev & 63] = true;
    }
    rb::launch_pdl(refiner_block_c144_split_kernel, dim3(p.total_tiles < sms ? p.total_tiles : sms), dim3(FS_THREADS), FS_SMEM, st, map_w[0], map_w[1], map_in, map_out, p);
    return check_launch("refiner_block_c144_split");
}

extern "C" int romab200_refiner_block_c144(const rb_refiner_block_c144_args* a, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    RB_REQUIRE(a->c == FZ_C, "refiner_block_c144: C must be 144 (got %d)", a->c);
    RB_REQUIRE(a->dtype == RB_F16 || a->dtype == RB_BF16 || a->dtype == RB_F32, "refiner_block_c144: fp16 / bf16 / fp32 activations");
    RB_REQUIRE(a->ld_pw % 8 == 0 && a->ld_pw >= FZ_C && ((uintptr_t)a->pw_weight) % 16 == 0, "refiner_block_c144: bad weight layout");
    static EncodeTiledFnFz enc = nullptr;
    if (!enc) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        RB_REQUIRE(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess && ptr,
                   "refiner_block_c144: cuTensorMapEncodeTiled not available");
        enc = (EncodeTiledFnFz)ptr;
    }
    if (a->dtype == RB_F32) return refiner_block_c144_split(a, st, enc);
    RB_REQUIRE(a->ld % 8 == 0 && a->ld >= FZ_C && ((uintptr_t)a->in) % 16 == 0 && ((uintptr_t)a->out) % 16 == 0 && a->in != a->out,
               "refiner_block_c144: bad activation layout");
    CUtensorMap map;
    cuuint64_t dims[2] = {(cuuint64_t)FZ_C, (cuuint64_t)FZ_C};
    cuuint64_t strides[1] = {(cuuint64_t)a->ld_pw * 2};
    cuuint32_t box[2] = {64, (cuuint32_t)FZ_C};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(&map, a->dtype == RB_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(a->pw_weight),
                     dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    RB_REQUIRE(r == CUDA_SUCCESS, "refiner_block_c144: cuTensorMapEncodeTiled failed with %d", (int)r);
    CUtensorMap map_in;          // activation [B, H, W, C] with pitch ld: box = 12 x 20 pixels x 144 channels, borders zero-filled
    {
        cuuint64_t d4[4] = {(cuuint64_t)FZ_C, (cuuint64_t)a->w, (cuuint64_t)a->h, (cuuint64_t)a->batch};
        cuuint64_t s4[3] = {(cuuint64_t)a->ld * 2, (cuuint64_t)a->w * a->ld * 2, (cuuint64_t)a->h * a->w * a->ld * 2};
        cuuint32_t b4[4] = {(cuuint32_t)FZ_C, (cuuint32_t)FZ_IW, (cuuint32_t)FZ_IH, 1};
        cuuint32_t e4[4] = {1, 1, 1, 1};
        CUresult r4 = enc(&map_in, a->dtype == RB_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(a->in),
                          d4, s4, b4, e4, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        RB_REQUIRE(r4 == CUDA_SUCCESS, "refiner_block_c144: cuTensorMapEncodeTiled (input) failed with %d", (int)r4);
    }
    FusedParams p;
    p.in = a->in; p.out = a->out; p.ld = a->ld; p.dw_w = a->dw_weight; p.ldw = a->ldw; p.dw_b = a->dw_bias; p.pw_b = a->pw_bias;
    p.batch = a->batch; p.H = a->h; p.W = a->w; p.tiles_x = (a->w + FZ_TW - 1) / FZ_TW; p.tiles_y = (a->h + FZ_TH - 1) / FZ_TH;
    const long long total = (long long)p.tiles_x * p.tiles_y * a->batch;
    RB_REQUIRE(total > 0 && total < (1ll << 31), "refiner_block_c144: bad tile count");
    p.total_tiles = (int)total; p.is_bf16 = a->dtype == RB_BF16;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int grid = p.total_tiles < sms ? p.total_tiles : sms;
    if (a->dtype == RB_F16) {
        static bool cfg[64] = {};            // function attributes are per device
        if (!cfg[dev & 63]) { RB_REQUIRE(cudaFuncSetAttribute(refiner_block_c144_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, FZ_SMEM) == cudaSuccess, "refiner_block_c144: smem attribute"); cfg[dev & 63] = true; }
        rb::launch_pdl(refiner_block_c144_kernel<__half>, dim3(grid), dim3(FZ_THREADS), FZ_SMEM, st, map, map_in, p);
    } else {
        static bool cfg[64] = {};
        if (!cfg[dev & 63]) { RB_REQUIRE(cudaFuncSetAttribute(refiner_block_c144_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, FZ_SMEM) == cudaSuccess, "refiner_block_c144: smem attribute"); cfg[dev & 63] = true; }
        rb::launch_pdl(refiner_block_c144_kernel<__nv_bfloat16>, dim3(grid), dim3(FZ_THREADS), FZ_SMEM, st, map, map_in, p);
    }
    return check_launch("refiner_block_c144");
}
