// Encoder convolutions on the 5th-generation tensor cores (sm_100a): implicit GEMM, forward.
//
// Replaces the cuDNN calls behind `torch.nn.Conv2d` in the reference's encoder
// (src/models/resnet_modified.py:40 stem, :126-134 conv3x3/conv1x1, used at :95-120, :159-177):
// 3x3 (and 1x1 downsample) convolutions, no bias, circular padding along the image width
// (CircularPad / F.pad(mode='circular'), :97,:100,:162,:167), zero padding along the height
// (padding=(1,0)), strides (1,1), (1,2), (2,2), followed by tanh / relu and, for the second conv
// of a BasicBlock, the residual add before the activation (:174-175).
//
// Layout: activations are NHWC bf16 with the padding MATERIALISED: [B, H+2, W+2, C]; rows 0 and
// H+1 are zero, column 0 is a copy of column W and column W+1 a copy of column 1 (the epilogue of
// the producing kernel writes both copies), so every filter tap of an output tile is a plain
// shifted box of the same tensor -> one TMA load per tap and K-chunk, no im2col buffer:
//     GEMM  M = 128 output pixels (TW along w x TH along h),  N = BN output channels,
//           K = taps x Cin, walked as (tap, 64-channel chunk).
// A (pixels x 64 ch) and B (BN filters x 64 ch) tiles are K-major, 128-byte swizzled, written by
// TMA (cp.async.bulk.tensor) into a 4-stage shared-memory ring; one elected thread issues
// tcgen05.mma (M=128, N=BN, K=16, bf16 -> fp32) with the accumulator in tensor memory;
// tcgen05.commit releases the stage; four epilogue warps read their TMEM lane quarter with
// tcgen05.ld, add the residual, apply the activation, convert to bf16 and store NHWC (plus the
// circular halo columns).  Warp roles: 0 = TMA producer, 1 = MMA issuer + TMEM allocator,
// 2..5 = epilogue.
#include <stdlib.h>
#include <cuda_fp16.h>
#include "tc_common.cuh"

namespace delora {

constexpr int kConvThreads = 192;
constexpr int kBlockM = 128;
constexpr int kBlockK = 64;           // bf16 elements = 128 bytes = one swizzle row
constexpr int kMaxStages = 4;         // smem ring depth is chosen per launch so that two CTAs fit on one SM
constexpr int kUmmaK = 16;

struct ConvParams {
    int B, Hout, Wout, Cin, Cout;
    int taps, ksize;                  // 9/3 or 1/1
    int stride_h, stride_w;
    int pad_off;                      // 0 for 3x3 (tap offset starts at padded coord 0), 1 for 1x1
    int TW, TH;                       // output tile: TW x TH = 128 pixels
    int tiles_w, tiles_h;             // tiles per image row / column
    int BN;
    int act;                          // 0 none, 1 relu, 2 tanh
    int stages;                       // smem ring depth (<= kMaxStages)
};

// ---------------------------------------------------------------- the kernel
__global__ void __launch_bounds__(kConvThreads, 2)
conv_fprop_tc_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w,
                     const __nv_bfloat16* __restrict__ residual, const __nv_bfloat16* __restrict__ saved,
                     __nv_bfloat16* __restrict__ y, ConvParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // 1024-byte alignment for the 128B swizzle atoms
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const int a_bytes = kBlockM * kBlockK * 2;            // 16 KB
    const int b_bytes = p.BN * kBlockK * 2;
    const int kStages = p.stages;
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem + kStages * a_bytes;
    uint64_t* full_bar = (uint64_t*)(smem_b + kStages * b_bytes);
    uint64_t* empty_bar = full_bar + kMaxStages;
    uint64_t* tmem_full_bar = empty_bar + kMaxStages;
    uint32_t* tmem_ptr_smem = (uint32_t*)(tmem_full_bar + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // tile coordinates: blockIdx.x -> (b, tile_h, tile_w), blockIdx.y -> n tile
    int t = blockIdx.x;
    const int tw_i = t % p.tiles_w; t /= p.tiles_w;
    const int th_i = t % p.tiles_h; t /= p.tiles_h;
    const int b = t;
    const int wo0 = tw_i * p.TW, ho0 = th_i * p.TH;
    const int n0 = blockIdx.y * p.BN;
    const int kchunks = p.Cin / kBlockK;
    const int n_iter = p.taps * kchunks;

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(full_bar + s, 1); mbar_init(empty_bar + s, 1); }
        mbar_init(tmem_full_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {   // allocate BN TMEM columns (power of two >= 32)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)),
                     "r"((uint32_t)p.BN));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_ptr_smem;

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w) : "memory");
            for (int it = 0; it < n_iter; ++it) {
                const int s = it % kStages;
                const uint32_t ph = (it / kStages) & 1;
                mbar_wait(empty_bar + s, ph ^ 1);
                const int tap = it / kchunks, kc = it - tap * kchunks;
                const int r = tap / p.ksize, q = tap - r * p.ksize;
                mbar_expect_tx(full_bar + s, (uint32_t)(a_bytes + b_bytes));
                tma_load_4d(smem_a + s * a_bytes, &map_x, full_bar + s, kc * kBlockK, wo0 * p.stride_w + q + p.pad_off,
                            ho0 * p.stride_h + r + p.pad_off, b);
                tma_load_2d(smem_b + s * b_bytes, &map_w, full_bar + s, tap * p.Cin + kc * kBlockK, n0);
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        // instruction descriptor: D = F32, A = B = BF16, both K-major, N = BN, M = 128
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.BN >> 3) << 17) |
                               ((uint32_t)(kBlockM >> 4) << 24);
        for (int it = 0; it < n_iter; ++it) {
            const int s = it % kStages;
            const uint32_t ph = (it / kStages) & 1;
            mbar_wait(full_bar + s, ph);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (lane == 0) {
                const uint64_t da = make_smem_desc(smem_u32(smem_a + s * a_bytes));
                const uint64_t db = make_smem_desc(smem_u32(smem_b + s * b_bytes));
#pragma unroll
                for (int k = 0; k < kBlockK / kUmmaK; ++k) {
                    // advance 16 bf16 = 32 bytes along K inside the swizzle row: +2 in 16-byte units
                    tcgen05_mma_bf16(tmem_base, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc,
                                     (it > 0 || k > 0) ? 1u : 0u);
                }
                tcgen05_commit(empty_bar + s);                       // frees the smem stage when the MMAs retire
                if (it == n_iter - 1) tcgen05_commit(tmem_full_bar); // accumulator complete
            }
            __syncwarp();
        }
    } else {
        // ===================== epilogue warps 2..5 =====================
        const int quarter = warp & 3;                                // TMEM lanes 32*quarter .. +31
        mbar_wait(tmem_full_bar, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int m = quarter * 32 + lane;                           // row of the tile = output pixel
        const int wo = wo0 + (m % p.TW), ho = ho0 + (m / p.TW);
        const bool in_range = (wo < p.Wout) && (ho < p.Hout);
        const int Wp = p.Wout + 2, Hp = p.Hout + 2;
        const size_t pix = ((size_t)b * Hp + (ho + 1)) * Wp + (wo + 1);
        for (int c0 = 0; c0 < p.BN; c0 += 32) {
            uint32_t acc[32];
            tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)c0, acc);
            if (in_range) {
                float v[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(acc[j]);
                if (residual) {
                    const uint4* rp = reinterpret_cast<const uint4*>(residual + pix * p.Cout + n0 + c0);
#pragma unroll
                    for (int j4 = 0; j4 < 4; ++j4) {
                        const uint4 rv = __ldg(rp + j4);
                        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&rv);
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const float2 f = __bfloat1622float2(h[e]);
                            v[j4 * 8 + e * 2] += f.x; v[j4 * 8 + e * 2 + 1] += f.y;
                        }
                    }
                }
                if (p.act >= 3) {
                    // backward (dgrad) modes: the accumulator is dL/d(activation output); multiply by the
                    // activation derivative evaluated on the SAVED forward output a: tanh' = 1 - a^2, relu' = [a > 0]
                    const uint4* sp = reinterpret_cast<const uint4*>(saved + pix * p.Cout + n0 + c0);
#pragma unroll
                    for (int j4 = 0; j4 < 4; ++j4) {
                        const uint4 sv = __ldg(sp + j4);
                        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&sv);
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const float2 a = __bfloat1622float2(h[e]);
                            const float d0 = (p.act == 3) ? fmaf(-a.x, a.x, 1.0f) : (a.x > 0.0f ? 1.0f : 0.0f);
                            const float d1 = (p.act == 3) ? fmaf(-a.y, a.y, 1.0f) : (a.y > 0.0f ? 1.0f : 0.0f);
                            v[j4 * 8 + e * 2] *= d0; v[j4 * 8 + e * 2 + 1] *= d1;
                        }
                    }
                }
                uint4 out[4];
#pragma unroll
                for (int j4 = 0; j4 < 4; ++j4) {
                    __nv_bfloat162 h[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e)
                        h[e] = __floats2bfloat162_rn(apply_act(v[j4 * 8 + e * 2], p.act), apply_act(v[j4 * 8 + e * 2 + 1], p.act));
                    out[j4] = *reinterpret_cast<uint4*>(h);
                }
                uint4* yp = reinterpret_cast<uint4*>(y + pix * p.Cout + n0 + c0);
#pragma unroll
                for (int j4 = 0; j4 < 4; ++j4) yp[j4] = out[j4];
                // circular halo columns of the padded output (read by the next layer's taps)
                if (wo == 0) {
                    uint4* hp = reinterpret_cast<uint4*>(y + (pix + p.Wout) * p.Cout + n0 + c0);
#pragma unroll
                    for (int j4 = 0; j4 < 4; ++j4) hp[j4] = out[j4];
                }
                if (wo == p.Wout - 1) {
                    uint4* hp = reinterpret_cast<uint4*>(y + (pix - p.Wout) * p.Cout + n0 + c0);
#pragma unroll
                    for (int j4 = 0; j4 < 4; ++j4) hp[j4] = out[j4];
                }
            }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    }
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.BN));
    }
}

// ---------------------------------------------------------------- weight gradient
// dW[co][tap][ci] = sum over output pixels of dZ[pix][co] * X[pix*stride + tap][ci]
// (autograd's backward of the reference's torch.nn.Conv2d layers, src/models/resnet_modified.py:40,:126-134).
// GEMM with M = output channels (128 per CTA), N = input channels (64..256 per CTA), K = PIXELS: both
// operands are pixel-major NHWC tiles (64 pixels x 64 channels, 128-byte rows, TMA SWIZZLE_128B), i.e.
// "MN-major" for the tensor core (a_major = b_major = 1 in the instruction descriptor; descriptor
// LBO = 8 KB between 64-channel blocks, SBO = 1 KB between groups of 8 pixel rows; one tcgen05.mma
// consumes K = 16 pixels = 2 KB).  One CTA = a GROUP of filter taps of one filter row x one (co, ci) tile x one
// slice of the pixels (split-K).  The kernel is bound by L2 -> shared-memory traffic (both operands stream, no
// reuse inside a tap), so for narrow layers the taps (r, q0..q0+tg-1) share the dZ tile: their shifted x boxes are
// stacked along N (Cin = 64: 3 taps, N = 192; Cin = 128: 2 taps, N = 256) -- 1.5x / 1.2x less traffic.  Each slice
// writes its fp32 partial, a second kernel sums the slices in a fixed order (deterministic) into the torch
// weight layout.
struct WgradParams {
    int B, Hout, Wout, Cin, Cout;
    int ksize, taps, stride_h, stride_w, pad_off;
    int TW, TH;               // a K tile = TW x TH = 64 output pixels
    int tiles_per_row;        // Wout / TW
    int row_tiles;            // Hout / TH
    int k_tiles;              // B * row_tiles * tiles_per_row
    int splits;
    int ci_tiles, nb;         // nb = 64-channel blocks of the N tile (N = 64 * nb)
    int a_blocks;             // 2 (Cout >= 128) or 1 (Cout == 64: rows 64..127 of the tile are unused)
    int stages;
    int tg;                   // filter taps (along the row, q) that share one CTA: their x boxes are stacked along N
    int groups_per_row;       // ceil(ksize / tg); grid.x = ksize * groups_per_row
};

__global__ void __launch_bounds__(kConvThreads, 1)
conv_wgrad_tc_kernel(const __grid_constant__ CUtensorMap map_dz, const __grid_constant__ CUtensorMap map_x,
                     float* __restrict__ partial, WgradParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const int blk_bytes = 64 * 64 * 2;                        // 64 pixels x 64 channels bf16 = 8 KB
    const int a_bytes = 2 * blk_bytes, b_bytes = p.tg * p.nb * blk_bytes;
    const int kStages = p.stages;
    uint8_t* smem_a = smem;
    uint8_t* smem_b = smem + kStages * a_bytes;
    uint64_t* full_bar = (uint64_t*)(smem_b + kStages * b_bytes);
    uint64_t* empty_bar = full_bar + kMaxStages;
    uint64_t* tmem_full_bar = empty_bar + kMaxStages;
    uint32_t* tmem_ptr_smem = (uint32_t*)(tmem_full_bar + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = blockIdx.x / p.groups_per_row, q0 = (blockIdx.x % p.groups_per_row) * p.tg;
    const int nq = min(p.tg, p.ksize - q0);                 // taps of this group: (r, q0 .. q0 + nq - 1)
    const int co_tile = blockIdx.y / p.ci_tiles, ci_tile = blockIdx.y % p.ci_tiles;
    const int split = blockIdx.z;
    const int co0 = co_tile * 128, ci0 = ci_tile * 64 * p.nb;
    const int per = (p.k_tiles + p.splits - 1) / p.splits;
    const int k_begin = split * per, k_end = min(p.k_tiles, k_begin + per);
    const int n_iter = max(0, k_end - k_begin);
    const int N = 64 * p.nb * nq;
    const uint32_t tmem_cols = N <= 64 ? 64u : (N <= 128 ? 128u : 256u);

    if (threadIdx.x == 0) {
        for (int s = 0; s < kMaxStages; ++s) { mbar_init(full_bar + s, 1); mbar_init(empty_bar + s, 1); }
        mbar_init(tmem_full_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)),
                     "r"(tmem_cols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_ptr_smem;

    if (warp == 0) {
        if (lane == 0) {
            for (int it = 0; it < n_iter; ++it) {
                const int s = it % kStages;
                const uint32_t ph = (it / kStages) & 1;
                mbar_wait(empty_bar + s, ph ^ 1);
                int kt = k_begin + it;
                const int wt = kt % p.tiles_per_row; kt /= p.tiles_per_row;
                const int ho = (kt % p.row_tiles) * p.TH;
                const int b = kt / p.row_tiles;
                mbar_expect_tx(full_bar + s, (uint32_t)((p.a_blocks + nq * p.nb) * blk_bytes));
                for (int j = 0; j < p.a_blocks; ++j)
                    tma_load_4d(smem_a + s * a_bytes + j * blk_bytes, &map_dz, full_bar + s, co0 + 64 * j, wt * p.TW + 1,
                                ho + 1, b);
                for (int t = 0; t < nq; ++t)
                    for (int j = 0; j < p.nb; ++j)
                        tma_load_4d(smem_b + s * b_bytes + (t * p.nb + j) * blk_bytes, &map_x, full_bar + s, ci0 + 64 * j,
                                    wt * p.TW * p.stride_w + q0 + t + p.pad_off, ho * p.stride_h + r + p.pad_off, b);
            }
        }
    } else if (warp == 1) {
        // D = F32, A = B = BF16, both MN-major (bits 15, 16), N, M = 128
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) |
                               ((uint32_t)(N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
        for (int it = 0; it < n_iter; ++it) {
            const int s = it % kStages;
            const uint32_t ph = (it / kStages) & 1;
            mbar_wait(full_bar + s, ph);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (lane == 0) {
                // MN-major SW128 descriptors: LBO = 8 KB (next 64-channel block), SBO = 1 KB (next 8 pixels)
                const uint32_t a_addr = smem_u32(smem_a + s * a_bytes), b_addr = smem_u32(smem_b + s * b_bytes);
#pragma unroll
                for (int k = 0; k < 4; ++k) {                 // 64 pixels = 4 x K16
                    uint64_t da = 0, db = 0;
                    da |= (uint64_t)(((a_addr + k * 2048) & 0x3FFFFu) >> 4);
                    da |= (uint64_t)(blk_bytes >> 4) << 16;
                    da |= (uint64_t)(1024 >> 4) << 32;
                    da |= (uint64_t)1 << 46;
                    da |= (uint64_t)2 << 61;
                    db |= (uint64_t)(((b_addr + k * 2048) & 0x3FFFFu) >> 4);
                    db |= (uint64_t)(blk_bytes >> 4) << 16;
                    db |= (uint64_t)(1024 >> 4) << 32;
                    db |= (uint64_t)1 << 46;
                    db |= (uint64_t)2 << 61;
                    tcgen05_mma_bf16(tmem_base, da, db, idesc, (it > 0 || k > 0) ? 1u : 0u);
                }
                tcgen05_commit(empty_bar + s);
                if (it == n_iter - 1) tcgen05_commit(tmem_full_bar);
            }
            __syncwarp();
        }
    } else {
        const int quarter = warp & 3;
        const int m = quarter * 32 + lane;                           // output channel row of the tile
        const int co = co0 + m;
        // accumulator column c -> (tap q0 + c / (64 nb), input channel ci0 + c % (64 nb))
        const int cols_per_tap = 64 * p.nb;
        if (n_iter > 0) {
            mbar_wait(tmem_full_bar, 0);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            for (int c0 = 0; c0 < N; c0 += 32) {
                uint32_t acc[32];
                tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)c0, acc);
                if (co < p.Cout) {
                    const int tap = r * p.ksize + q0 + c0 / cols_per_tap;
                    float* __restrict__ out = partial + (((size_t)split * p.taps + tap) * p.Cout + co) * p.Cin + ci0 +
                                              c0 % cols_per_tap;
                    float4* o4 = reinterpret_cast<float4*>(out);
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        o4[j] = make_float4(__uint_as_float(acc[4 * j]), __uint_as_float(acc[4 * j + 1]),
                                            __uint_as_float(acc[4 * j + 2]), __uint_as_float(acc[4 * j + 3]));
                }
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        } else if (co < p.Cout) {
            for (int c = 0; c < N; ++c) {
                const int tap = r * p.ksize + q0 + c / cols_per_tap;
                partial[(((size_t)split * p.taps + tap) * p.Cout + co) * p.Cin + ci0 + c % cols_per_tap] = 0.0f;
            }
        }
    }
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols));
    }
}

// sum the split-K slices in order and write the torch layout dW[co][ci][r][s] (ci < Cin_true)
__global__ void __launch_bounds__(256)
wgrad_reduce_kernel(const float* __restrict__ partial, int splits, int taps, int Cout, int Cin, int Cin_true,
                    float* __restrict__ dw) {
    const size_t total = (size_t)Cout * Cin_true * taps;
    const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= total) return;
    const int tap = (int)(i % taps);
    const int ci = (int)((i / taps) % Cin_true);
    const int co = (int)(i / ((size_t)taps * Cin_true));
    float acc = 0.0f;
    for (int s = 0; s < splits; ++s) acc += partial[(((size_t)s * taps + tap) * Cout + co) * Cin + ci];
    dw[i] = acc;
}

// ---------------------------------------------------------------- layout helpers (bandwidth kernels)
// two [B,4,H,W] fp32 range images -> [B, H+2, W+2, Cpad] bf16, channels 0..7 = cat(image_1, image_2)
// (src/models/model.py:98), the rest zero; circular halo columns, zero halo rows.
__global__ void __launch_bounds__(256)
images_to_nhwc_kernel(const float* __restrict__ img1, const float* __restrict__ img2, int B, int H, int W, int Cpad,
                      __nv_bfloat16* __restrict__ x) {
    // one thread per (padded pixel, group of 8 channels): 16-byte stores, a pixel's Cpad channels are
    // written by Cpad/8 adjacent threads (coalesced); only group 0 carries data (8 real channels)
    const int Wp = W + 2, Hp = H + 2, groups = Cpad / 8;
    const size_t total = (size_t)B * Hp * Wp * groups;
    const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= total) return;
    const int grp = (int)(i % groups);
    const size_t pixel = i / groups;
    const int wp = (int)(pixel % Wp), hp = (int)((pixel / Wp) % Hp), b = (int)(pixel / ((size_t)Wp * Hp));
    uint4 out = make_uint4(0u, 0u, 0u, 0u);
    if (grp == 0 && hp != 0 && hp != Hp - 1) {
        int w = wp - 1;
        if (w < 0) w = W - 1;
        if (w >= W) w = 0;
        const int h = hp - 1;
        __nv_bfloat162 v[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const float* src = (c < 2) ? img1 : img2;
            const size_t base = (((size_t)b * 4 + (2 * c & 3)) * H + h) * W + w;
            v[c] = __floats2bfloat162_rn(__ldg(src + base), __ldg(src + base + (size_t)H * W));
        }
        out = *reinterpret_cast<uint4*>(v);
    }
    *reinterpret_cast<uint4*>(x + pixel * Cpad + grp * 8) = out;
}

// MaxPool2d(3, stride (1,2), padding (1,0)) after circular W padding (src/models/resnet_modified.py:46,:100-101),
// NHWC padded in / out; the height padding of the pool is -inf (PyTorch), i.e. rows outside are skipped.
__global__ void __launch_bounds__(256)
maxpool_nhwc_kernel(const __nv_bfloat16* __restrict__ x, int B, int H, int W, int C, __nv_bfloat16* __restrict__ y) {
    const int Wout = W / 2;
    const size_t total = (size_t)B * H * Wout * (C / 2);
    const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= total) return;
    const int c2 = (int)(i % (C / 2));
    size_t r = i / (C / 2);
    const int wo = (int)(r % Wout); r /= Wout;
    const int ho = (int)(r % H);
    const int b = (int)(r / H);
    const int Wp = W + 2, Hp = H + 2, Wpo = Wout + 2;
    float m0 = -INFINITY, m1 = -INFINITY;
    for (int dr = -1; dr <= 1; ++dr) {
        const int h = ho + dr;
        if (h < 0 || h >= H) continue;
        for (int dq = 0; dq < 3; ++dq) {
            const int wp = 2 * wo + dq;                  // padded column index (circular halo materialised)
            const __nv_bfloat162 v = *reinterpret_cast<const __nv_bfloat162*>(
                x + (((size_t)b * Hp + h + 1) * Wp + wp) * C + 2 * c2);
            const float2 f = __bfloat1622float2(v);
            m0 = fmaxf(m0, f.x); m1 = fmaxf(m1, f.y);
        }
    }
    const __nv_bfloat162 o = __floats2bfloat162_rn(m0, m1);
    const size_t pix = ((size_t)b * Hp + ho + 1) * Wpo + wo + 1;
    *reinterpret_cast<__nv_bfloat162*>(y + pix * C + 2 * c2) = o;
    if (wo == 0) *reinterpret_cast<__nv_bfloat162*>(y + (pix + Wout) * C + 2 * c2) = o;
    if (wo == Wout - 1) *reinterpret_cast<__nv_bfloat162*>(y + (pix - Wout) * C + 2 * c2) = o;
}

// Backward of a strided convolution = stride-1 convolution of the ZERO-UPSAMPLED output gradient with the
// flipped filter.  x [B,H+2,W+2,C] padded -> y [B,H*sh+2,W*sw+2,C] padded: y[h*sh, w*sw] = x[h, w], zeros
// elsewhere (incl. correct circular halo columns and zero halo rows).
__global__ void __launch_bounds__(256)
zero_upsample_kernel(const __nv_bfloat16* __restrict__ x, int B, int H, int W, int C, int sh, int sw, int Ho, int Wo,
                     __nv_bfloat16* __restrict__ y) {
    const int groups = C / 8;
    const size_t total = (size_t)B * (Ho + 2) * (Wo + 2) * groups;
    const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= total) return;
    const int g = (int)(i % groups);
    const size_t pixel = i / groups;
    const int wp = (int)(pixel % (Wo + 2)), hp = (int)((pixel / (Wo + 2)) % (Ho + 2));
    const int b = (int)(pixel / ((size_t)(Wo + 2) * (Ho + 2)));
    uint4 out = make_uint4(0u, 0u, 0u, 0u);
    if (hp >= 1 && hp <= Ho) {
        int w = wp - 1;                       // circular halo: padded col 0 = col Wo-1, col Wo+1 = col 0
        if (w < 0) w = Wo - 1;
        if (w >= Wo) w = 0;
        const int h = hp - 1;
        if (h % sh == 0 && w % sw == 0 && h / sh < H && w / sw < W)
            out = __ldg(reinterpret_cast<const uint4*>(x + ((((size_t)b * (H + 2)) + h / sh + 1) * (W + 2) + w / sw + 1) * C) + g);
    }
    *reinterpret_cast<uint4*>(y + pixel * C + g * 8) = out;
}

// Max-pool with argmax (training): same window as maxpool_nhwc_kernel, additionally stores which of the 9
// window positions won (first maximum in (row, column) scan order, as PyTorch's backward assumes).
// `act` != 0: x holds PRE-activations z and the output is act(max z) = max act(z) (tanh / relu are monotonic), so the
// backward can evaluate act'(z) from z itself -- 1 - a^2 from a bf16-rounded, saturated a = tanh(z) has no correct digit.
__global__ void __launch_bounds__(256)
maxpool_idx_nhwc_kernel(const __nv_bfloat16* __restrict__ x, int B, int H, int W, int C, __nv_bfloat16* __restrict__ y,
                        uint8_t* __restrict__ idx, int act, int in_f16) {
    // one thread = 8 channels of one output pixel: 16-byte loads / stores, 8-byte argmax store
    const int Wout = W / 2, groups = C / 8;
    const size_t total = (size_t)B * H * Wout * groups;
    const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= total) return;
    const int grp = (int)(i % groups);
    size_t r = i / groups;
    const int wo = (int)(r % Wout); r /= Wout;
    const int ho = (int)(r % H);
    const int b = (int)(r / H);
    const int Wp = W + 2, Hp = H + 2, Wpo = Wout + 2;
    float m[8];
    int arg[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) { m[e] = -INFINITY; arg[e] = 4; }
#pragma unroll
    for (int dr = 0; dr < 3; ++dr) {
        const int h = ho + dr - 1;
        if (h < 0 || h >= H) continue;
#pragma unroll
        for (int dq = 0; dq < 3; ++dq) {
            const uint4 raw = __ldg(reinterpret_cast<const uint4*>(x + (((size_t)b * Hp + h + 1) * Wp + 2 * wo + dq) * C) + grp);
            const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&raw);
            const __half2* g2 = reinterpret_cast<const __half2*>(&raw);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float2 f = in_f16 ? __half22float2(g2[e]) : __bfloat1622float2(h2[e]);
                if (f.x > m[2 * e]) { m[2 * e] = f.x; arg[2 * e] = dr * 3 + dq; }
                if (f.y > m[2 * e + 1]) { m[2 * e + 1] = f.y; arg[2 * e + 1] = dr * 3 + dq; }
            }
        }
    }
    __nv_bfloat162 o2[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) o2[e] = __floats2bfloat162_rn(apply_act(m[2 * e], act), apply_act(m[2 * e + 1], act));
    const uint4 out = *reinterpret_cast<uint4*>(o2);
    const size_t pix = ((size_t)b * Hp + ho + 1) * Wpo + wo + 1;
    reinterpret_cast<uint4*>(y + pix * C)[grp] = out;
    if (wo == 0) reinterpret_cast<uint4*>(y + (pix + Wout) * C)[grp] = out;
    if (wo == Wout - 1) reinterpret_cast<uint4*>(y + (pix - Wout) * C)[grp] = out;
    uint2 packed;
    packed.x = (unsigned)arg[0] | ((unsigned)arg[1] << 8) | ((unsigned)arg[2] << 16) | ((unsigned)arg[3] << 24);
    packed.y = (unsigned)arg[4] | ((unsigned)arg[5] << 8) | ((unsigned)arg[6] << 16) | ((unsigned)arg[7] << 24);
    reinterpret_cast<uint2*>(idx + ((((size_t)b * H + ho) * Wout + wo) * C))[grp] = packed;
}

// Backward of that pool fused with the derivative of the activation that produced its input:
// dz[b,h,w,c] = act'(a[b,h,w,c]) * sum of dy over the (<= 6) windows whose argmax is (h, w).
// w is an UNPADDED input column; the windows see the circularly padded row, so padded column 0 / W+1
// alias columns W-1 / 0.  Output dz is padded NHWC with halo (it feeds the stem's wgrad).
__global__ void __launch_bounds__(256)
maxpool_bwd_act_kernel(const __nv_bfloat16* __restrict__ dy, const uint8_t* __restrict__ idx,
                       const __nv_bfloat16* __restrict__ a, int B, int H, int W, int C, int act,
                       __nv_bfloat16* __restrict__ dz, int a_f16) {
    // one thread = 8 channels of one input pixel (16-byte accesses)
    const int Wout = W / 2, groups = C / 8;
    const size_t total = (size_t)B * H * W * groups;
    const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= total) return;
    const int grp = (int)(i % groups);
    size_t r = i / groups;
    const int w = (int)(r % W); r /= W;
    const int h = (int)(r % H);
    const int b = (int)(r / H);
    const int Wp = W + 2, Hp = H + 2, Wpo = Wout + 2;
    float g[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) g[e] = 0.0f;
    // Windows that contain input column w: padded column wp = 2 wo + dq.  wp = w + 1 always; the circular halo adds
    // wp = 0 for w == W - 1 (wp = W + 1 for w == 0 would need wo = Wout: outside).  At most 3 (wo, dq) candidates x 3
    // rows = 9 windows; all argmax words are loaded first (independent 8-byte loads), then the matching dy rows.
    int c_wo[3], c_dq[3];
    int nc = 0;
    {
        const int wp = w + 1;
        if (wp & 1) { c_wo[nc] = (wp - 1) >> 1; c_dq[nc] = 1; ++nc; }
        else {
            c_wo[nc] = wp >> 1; c_dq[nc] = 0; ++nc;
            c_wo[nc] = (wp >> 1) - 1; c_dq[nc] = 2; ++nc;
        }
        if (w == W - 1) { c_wo[nc] = 0; c_dq[nc] = 0; ++nc; }              // halo copy at padded column 0
    }
    uint2 am[9];
    bool ok[9];
#pragma unroll
    for (int ci = 0; ci < 3; ++ci)
#pragma unroll
        for (int dr = 0; dr < 3; ++dr) {
            const int ho = h - dr + 1;
            const bool valid = ci < nc && ho >= 0 && ho < H && c_wo[ci < nc ? ci : 0] < Wout;
            ok[ci * 3 + dr] = valid;
            am[ci * 3 + dr] = valid ? __ldg(reinterpret_cast<const uint2*>(idx + (((size_t)b * H + ho) * Wout + c_wo[ci]) * C) + grp)
                                    : make_uint2(0xffffffffu, 0xffffffffu);
        }
#pragma unroll
    for (int ci = 0; ci < 3; ++ci)
#pragma unroll
        for (int dr = 0; dr < 3; ++dr) {
            if (!ok[ci * 3 + dr]) continue;
            const unsigned want = (unsigned)(dr * 3 + c_dq[ci]) * 0x01010101u;
            const unsigned eq_lo = am[ci * 3 + dr].x ^ want, eq_hi = am[ci * 3 + dr].y ^ want;   // zero byte = argmax is (h, w)
            if ((((eq_lo - 0x01010101u) & ~eq_lo) | ((eq_hi - 0x01010101u) & ~eq_hi)) & 0x80808080u) {
                const int ho = h - dr + 1;
                const uint4 raw = __ldg(reinterpret_cast<const uint4*>(dy + (((size_t)b * Hp + ho + 1) * Wpo + c_wo[ci] + 1) * C) + grp);
                const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float2 f = __bfloat1622float2(h2[e]);
                    const unsigned word = (e < 2) ? eq_lo : eq_hi;
                    if (((word >> (16 * (e & 1))) & 0xffu) == 0u) g[2 * e] += f.x;
                    if (((word >> (16 * (e & 1) + 8)) & 0xffu) == 0u) g[2 * e + 1] += f.y;
                }
            }
        }
    const uint4 araw = __ldg(reinterpret_cast<const uint4*>(a + (((size_t)b * Hp + h + 1) * Wp + w + 1) * C) + grp);
    const __nv_bfloat162* a2 = reinterpret_cast<const __nv_bfloat162*>(&araw);
    const __half2* a2h = reinterpret_cast<const __half2*>(&araw);
    __nv_bfloat162 o2[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const float2 av = a_f16 ? __half22float2(a2h[e]) : __bfloat1622float2(a2[e]);
        float d0, d1;
        if (act == 6) {            // `a` holds pre-activations z: tanh'(z) = 4 e / (1 + e)^2, e = exp(-2 |z|) (no cancellation)
            const float e0 = __expf(-2.0f * fabsf(av.x)), e1 = __expf(-2.0f * fabsf(av.y));
            d0 = __fdividef(4.0f * e0, (1.0f + e0) * (1.0f + e0));
            d1 = __fdividef(4.0f * e1, (1.0f + e1) * (1.0f + e1));
        } else {
            d0 = (act == 2) ? fmaf(-av.x, av.x, 1.0f) : ((act == 1 || act == 5) ? (av.x > 0.0f ? 1.0f : 0.0f) : 1.0f);
            d1 = (act == 2) ? fmaf(-av.y, av.y, 1.0f) : ((act == 1 || act == 5) ? (av.y > 0.0f ? 1.0f : 0.0f) : 1.0f);
        }
        o2[e] = __floats2bfloat162_rn(g[2 * e] * d0, g[2 * e + 1] * d1);
    }
    const uint4 out = *reinterpret_cast<uint4*>(o2);
    const size_t pix = ((size_t)b * Hp + h + 1) * Wp + w + 1;
    reinterpret_cast<uint4*>(dz + pix * C)[grp] = out;
    if (w == 0) reinterpret_cast<uint4*>(dz + (pix + W) * C)[grp] = out;
    if (w == W - 1) reinterpret_cast<uint4*>(dz + (pix - W) * C)[grp] = out;
}

// Tiled form of maxpool_bwd_act_kernel for C = 64, W % 32 == 0 (the stem's shape): a CTA owns 4 input rows x 32 input
// columns; the argmax bytes and dy rows of the (6 x 17 [+ the wrap window]) pooling windows that touch the tile are
// staged ONCE in shared memory (coalesced 8- / 16-byte loads), then every (pixel, 8-channel group) gathers its <= 9
// candidate windows from there in the same fixed order as the per-pixel kernel (bit-identical results, no atomics).
// The per-pixel kernel re-read each argmax word from L1/L2 nine times (283 us at B = 16, 64 x 1024 x 64).
constexpr int kPoolTH = 4, kPoolTW = 32;
__global__ void __launch_bounds__(256)
maxpool_bwd_tile_kernel(const __nv_bfloat16* __restrict__ dy, const uint8_t* __restrict__ idx,
                        const __nv_bfloat16* __restrict__ a, int B, int H, int W, int act,
                        __nv_bfloat16* __restrict__ dz, int a_f16) {
    constexpr int C = 64, G = 8, NR = kPoolTH + 2, NC = kPoolTW / 2 + 2;       // 6 window rows, 17 columns + wrap slot
    __shared__ uint2 s_idx[NR][NC][G];
    __shared__ uint4 s_dy[NR][NC][G];
    const int Wout = W / 2, Wp = W + 2, Hp = H + 2, Wpo = Wout + 2;
    const int w0 = blockIdx.x * kPoolTW, h0 = blockIdx.y * kPoolTH, b = blockIdx.z;
    const bool last_tile = (w0 + kPoolTW == W);
    for (int t = threadIdx.x; t < NR * NC * G; t += 256) {
        const int grp = t % G, wi = (t / G) % NC, ri = t / (G * NC);
        const int ho = h0 - 1 + ri;
        const int wo = (wi < NC - 1) ? (w0 >> 1) + wi : 0;                     // slot NC-1: the window at wo = 0 (circular halo)
        const bool valid = ho >= 0 && ho < H && wo < Wout && (wi < NC - 1 || last_tile);
        s_idx[ri][wi][grp] = valid ? __ldg(reinterpret_cast<const uint2*>(idx + (((size_t)b * H + ho) * Wout + wo) * C) + grp)
                                   : make_uint2(0xffffffffu, 0xffffffffu);
        s_dy[ri][wi][grp] = valid ? __ldg(reinterpret_cast<const uint4*>(dy + (((size_t)b * Hp + ho + 1) * Wpo + wo + 1) * C) + grp)
                                  : make_uint4(0u, 0u, 0u, 0u);
    }
    __syncthreads();
    for (int item = threadIdx.x; item < kPoolTH * kPoolTW * G; item += 256) {
        const int grp = item % G, lw = (item / G) % kPoolTW, lh = item / (G * kPoolTW);
        const int h = h0 + lh, w = w0 + lw;
        if (h >= H) continue;
        float g[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) g[e] = 0.0f;
        // candidate windows in the per-pixel kernel's order: (wo, dq) from padded column wp = w + 1, then the halo copy
        const int wp = w + 1, odd = wp & 1;
        const int c_wi[3] = {(odd ? (wp - 1) >> 1 : wp >> 1) - (w0 >> 1), (wp >> 1) - 1 - (w0 >> 1), NC - 1};
        const int c_dq[3] = {odd ? 1 : 0, 2, 0};
        const bool c_ok[3] = {true, !odd, w == W - 1};
#pragma unroll
        for (int ci = 0; ci < 3; ++ci) {
            if (!c_ok[ci]) continue;
#pragma unroll
            for (int dr = 0; dr < 3; ++dr) {
                const int ri = lh - dr + 2;                                    // window row ho = h - dr + 1
                const uint2 am = s_idx[ri][c_wi[ci]][grp];
                const unsigned want = (unsigned)(dr * 3 + c_dq[ci]) * 0x01010101u;
                const unsigned eq_lo = am.x ^ want, eq_hi = am.y ^ want;       // zero byte = this window's argmax is (h, w)
                if ((((eq_lo - 0x01010101u) & ~eq_lo) | ((eq_hi - 0x01010101u) & ~eq_hi)) & 0x80808080u) {
                    const uint4 raw = s_dy[ri][c_wi[ci]][grp];
                    const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const float2 f = __bfloat1622float2(h2[e]);
                        const unsigned word = (e < 2) ? eq_lo : eq_hi;
                        if (((word >> (16 * (e & 1))) & 0xffu) == 0u) g[2 * e] += f.x;
                        if (((word >> (16 * (e & 1) + 8)) & 0xffu) == 0u) g[2 * e + 1] += f.y;
                    }
                }
            }
        }
        const uint4 araw = __ldg(reinterpret_cast<const uint4*>(a + (((size_t)b * Hp + h + 1) * Wp + w + 1) * C) + grp);
        const __nv_bfloat162* a2 = reinterpret_cast<const __nv_bfloat162*>(&araw);
        const __half2* a2h = reinterpret_cast<const __half2*>(&araw);
        __nv_bfloat162 o2[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float2 av = a_f16 ? __half22float2(a2h[e]) : __bfloat1622float2(a2[e]);
            float d0, d1;
            if (act == 6) {
                const float e0 = __expf(-2.0f * fabsf(av.x)), e1 = __expf(-2.0f * fabsf(av.y));
                d0 = __fdividef(4.0f * e0, (1.0f + e0) * (1.0f + e0));
                d1 = __fdividef(4.0f * e1, (1.0f + e1) * (1.0f + e1));
            } else {
                d0 = (act == 2) ? fmaf(-av.x, av.x, 1.0f) : ((act == 1 || act == 5) ? (av.x > 0.0f ? 1.0f : 0.0f) : 1.0f);
                d1 = (act == 2) ? fmaf(-av.y, av.y, 1.0f) : ((act == 1 || act == 5) ? (av.y > 0.0f ? 1.0f : 0.0f) : 1.0f);
            }
            o2[e] = __floats2bfloat162_rn(g[2 * e] * d0, g[2 * e + 1] * d1);
        }
        const uint4 out = *reinterpret_cast<uint4*>(o2);
        const size_t pix = ((size_t)b * Hp + h + 1) * Wp + w + 1;
        reinterpret_cast<uint4*>(dz + pix * C)[grp] = out;
        if (w == 0) reinterpret_cast<uint4*>(dz + (pix + W) * C)[grp] = out;
        if (w == W - 1) reinterpret_cast<uint4*>(dz + (pix - W) * C)[grp] = out;
    }
}

// Backward of AdaptiveAvgPool2d((1,1)) fused with the derivative of the last block's activation:
// dz[b,h,w,c] = g[b,c] / (H*W) * act'(a[b,h,w,c]), padded NHWC with halo.
__global__ void __launch_bounds__(256)
avgpool_bwd_act_kernel(const float* __restrict__ g, const __nv_bfloat16* __restrict__ a, int B, int H, int W, int C,
                       int act, __nv_bfloat16* __restrict__ dz) {
    // one thread = 8 channels of one pixel (16-byte accesses)
    const int groups = C / 8;
    const size_t total = (size_t)B * H * W * groups;
    const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= total) return;
    const int grp = (int)(i % groups);
    size_t r = i / groups;
    const int w = (int)(r % W); r /= W;
    const int h = (int)(r % H);
    const int b = (int)(r / H);
    const size_t pix = ((size_t)b * (H + 2) + h + 1) * (W + 2) + w + 1;
    const uint4 araw = __ldg(reinterpret_cast<const uint4*>(a + pix * C) + grp);
    const __nv_bfloat162* a2 = reinterpret_cast<const __nv_bfloat162*>(&araw);
    const float4 g0 = __ldg(reinterpret_cast<const float4*>(g + (size_t)b * C + grp * 8));
    const float4 g1 = __ldg(reinterpret_cast<const float4*>(g + (size_t)b * C + grp * 8) + 1);
    const float gv[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
    const float inv = 1.0f / (float)(H * W);
    __nv_bfloat162 o2[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const float2 av = __bfloat1622float2(a2[e]);
        const float d0 = (act == 2) ? fmaf(-av.x, av.x, 1.0f) : (act == 1 ? (av.x > 0.0f ? 1.0f : 0.0f) : 1.0f);
        const float d1 = (act == 2) ? fmaf(-av.y, av.y, 1.0f) : (act == 1 ? (av.y > 0.0f ? 1.0f : 0.0f) : 1.0f);
        o2[e] = __floats2bfloat162_rn(gv[2 * e] * inv * d0, gv[2 * e + 1] * inv * d1);
    }
    const uint4 out = *reinterpret_cast<uint4*>(o2);
    reinterpret_cast<uint4*>(dz + pix * C)[grp] = out;
    if (w == 0) reinterpret_cast<uint4*>(dz + (pix + W) * C)[grp] = out;
    if (w == W - 1) reinterpret_cast<uint4*>(dz + (pix - W) * C)[grp] = out;
}

// AdaptiveAvgPool2d((1,1)) of the last feature map (src/models/resnet_modified.py:111): padded NHWC bf16 -> [B, C] fp32.
// One CTA = 64 channels of one image; 32 pixel lanes x 8 channel groups (16-byte loads, 128-byte runs per pixel),
// fp32 sums in a fixed order (deterministic), mean = sum / (H W).  Replaces slice -> .float() -> mean (two kernels,
// 50 MB of traffic for the 16.8 MB map at B = 16).
__global__ void __launch_bounds__(256)
avgpool_nhwc_kernel(const __nv_bfloat16* __restrict__ x, int H, int W, int C, float* __restrict__ y) {
    __shared__ float part[32][65];
    const int b = blockIdx.y, c0 = blockIdx.x * 64;
    const int grp = threadIdx.x & 7, pl = threadIdx.x >> 3;
    float s[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) s[e] = 0.0f;
    const int HW = H * W;
    for (int p = pl; p < HW; p += 32) {
        const int h = p / W, w = p - h * W;
        const size_t pix = ((size_t)b * (H + 2) + h + 1) * (W + 2) + w + 1;
        const uint4 raw = __ldg(reinterpret_cast<const uint4*>(x + pix * C + c0) + grp);
        const __nv_bfloat162* v2 = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float2 f = __bfloat1622float2(v2[e]);
            s[2 * e] += f.x; s[2 * e + 1] += f.y;
        }
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) part[pl][grp * 8 + e] = s[e];
    __syncthreads();
    if (threadIdx.x < 64) {
        float t = 0.0f;
#pragma unroll 8
        for (int k = 0; k < 32; ++k) t += part[k][threadIdx.x];
        y[(size_t)b * C + c0 + threadIdx.x] = t / (float)HW;
    }
}

// padded NHWC bf16 -> NCHW fp32 (interior only): the reference's feature-map layout, for checks / heads
__global__ void __launch_bounds__(256)
nhwc_to_nchw_kernel(const __nv_bfloat16* __restrict__ x, int B, int H, int W, int C, float* __restrict__ y) {
    const size_t total = (size_t)B * C * H * W;
    const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= total) return;
    const int w = (int)(i % W), h = (int)((i / W) % H), c = (int)((i / ((size_t)W * H)) % C);
    const int b = (int)(i / ((size_t)W * H * C));
    y[i] = __bfloat162float(x[(((size_t)b * (H + 2) + h + 1) * (W + 2) + w + 1) * C + c]);
}

// fp32 torch filter [Cout, Cin, k, k] -> the two bf16 layouts the convolution kernels read, in one launch:
//   w_fwd [Cout, k*k, Cin_pad]  (tap-major K of fprop; channels >= Cin zero)
//   w_flip[Cin,  k*k, Cout]     (filter of the data-gradient convolution: spatially flipped, in/out swapped)
__global__ void __launch_bounds__(256)
weight_prep_kernel(const float* __restrict__ w, int Cout, int Cin, int k, int Cin_pad, __nv_bfloat16* __restrict__ w_fwd,
                   __nv_bfloat16* __restrict__ w_flip) {
    const int taps = k * k;
    const size_t n_fwd = (size_t)Cout * taps * Cin_pad, n_flip = w_flip ? (size_t)Cin * taps * Cout : 0;
    const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (i < n_fwd) {
        const int ci = (int)(i % Cin_pad), tap = (int)((i / Cin_pad) % taps), co = (int)(i / ((size_t)Cin_pad * taps));
        w_fwd[i] = __float2bfloat16_rn(ci < Cin ? __ldg(w + ((size_t)co * Cin + ci) * taps + tap) : 0.0f);
    } else if (i < n_fwd + n_flip) {
        const size_t j = i - n_fwd;
        const int co = (int)(j % Cout), tap = (int)((j / Cout) % taps), ci = (int)(j / ((size_t)Cout * taps));
        w_flip[j] = __float2bfloat16_rn(__ldg(w + ((size_t)co * Cin + ci) * taps + (taps - 1 - tap)));
    }
}

// ---------------------------------------------------------------- host side
static PFN_cuTensorMapEncodeTiled_v12000 get_encode() { return get_tensor_map_encoder(); }

struct TensorMaps {
    CUtensorMap x, w;
};

// Output tile of `pixels` (128 fprop / 64 wgrad) = TW x TH with TW a power of two >= 4: the shape that wastes
// the fewest pixels on a Hout x Wout image (ragged tiles are zero-filled by TMA on the way in and masked
// on the way out), the widest one on ties.  64x2048 images tile exactly; KITTI's 64x720 (widths 360, 180,
// 90, 45, 23 down the encoder) pads by 0-7 %.
static void pick_tile(int Hout, int Wout, int pixels, int* TW, int* TH) {
    long best = -1;
    for (int tw = pixels; tw >= 4; tw >>= 1) {
        const int th = pixels / tw;
        if (th > 64) break;
        const long cost = (long)((Wout + tw - 1) / tw) * tw * (long)((Hout + th - 1) / th) * th;
        if (best < 0 || cost < best) { best = cost; *TW = tw; *TH = th; }
    }
}

// Tensor maps depend only on (pointers, shapes); encoding them costs a few microseconds of host time
// per call, which matters when 20 convolutions are launched back to back.  Small per-thread cache.
static const TensorMaps* get_maps(const void* x, const void* w, int B, int Hin, int Win, int Cin, int Cout,
                                  const ConvParams& p) {
    struct Key { const void* x; const void* w; int B, Hin, Win, Cin, Cout, ks, sh, sw; };
    struct Entry { Key k; TensorMaps m; };
    static thread_local Entry cache[64];
    static thread_local int used = 0, next = 0;
    const Key key = {x, w, B, Hin, Win, Cin, Cout, p.ksize, p.stride_h, p.stride_w};
    for (int i = 0; i < used; ++i) {
        const Key& c = cache[i].k;
        if (c.x == key.x && c.w == key.w && c.B == key.B && c.Hin == key.Hin && c.Win == key.Win && c.Cin == key.Cin &&
            c.Cout == key.Cout && c.ks == key.ks && c.sh == key.sh && c.sw == key.sw)
            return &cache[i].m;
    }
    PFN_cuTensorMapEncodeTiled_v12000 encode = get_encode();
    if (!encode) return nullptr;
    Entry& e = cache[next];
    const int Hp = Hin + 2, Wp = Win + 2;
    {
        cuuint64_t dims[4] = {(cuuint64_t)Cin, (cuuint64_t)Wp, (cuuint64_t)Hp, (cuuint64_t)B};
        cuuint64_t strides[3] = {(cuuint64_t)Cin * 2, (cuuint64_t)Wp * Cin * 2, (cuuint64_t)Hp * Wp * Cin * 2};
        // with a traversal stride the box spans TW*stride_w (TH*stride_h) elements and loads every stride-th one
        cuuint32_t box[4] = {(cuuint32_t)kBlockK, (cuuint32_t)(p.TW * p.stride_w), (cuuint32_t)(p.TH * p.stride_h), 1};
        cuuint32_t estr[4] = {1, (cuuint32_t)p.stride_w, (cuuint32_t)p.stride_h, 1};
        if (encode(&e.m.x, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(x), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return nullptr;
    }
    {
        cuuint64_t dims[2] = {(cuuint64_t)p.taps * Cin, (cuuint64_t)Cout};
        cuuint64_t strides[1] = {(cuuint64_t)p.taps * Cin * 2};
        cuuint32_t box[2] = {(cuuint32_t)kBlockK, (cuuint32_t)p.BN};
        cuuint32_t estr[2] = {1, 1};
        if (encode(&e.m.w, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(w), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return nullptr;
    }
    e.k = key;
    const TensorMaps* out = &e.m;
    next = (next + 1) % 64;
    if (used < 64) ++used;
    return out;
}

}  // namespace delora

namespace delora {
bool conv_rows_eligible(int Cin, int Cout, int ksize, int Wg);
void rows_set_pairs(int on);
bool rows_use_pairs();
bool wgrad2_eligible(int Cin, int Cout, int ksize, int stride_h, int stride_w);
int64_t wgrad2_scratch_floats(int B, int Hout, int Wout, int Cin, int Cout, int sw);
int wgrad2_launch(const void* x, const void* dz, float* dw, float* scratch, int B, int Hin, int Win, int Cin, int Cin_true,
                  int Cout, int stride_h, int stride_w, cudaStream_t st);
int conv_rows_launch(const void* x, const void* w, const void* residual, const void* saved, void* y, int B, int Hout,
                     int Wout, int Cin, int Cout, int ksize, int up_h, int up_w, int act, cudaStream_t stream,
                     int residual_on_grid);
// DELORA_CONV_ROWS=0 keeps every convolution on the first-generation kernel (A/B measurements)
static int g_conv_rows = -1;
static bool use_conv_rows() {
    if (g_conv_rows < 0) { const char* e = getenv("DELORA_CONV_ROWS"); g_conv_rows = (e && e[0] == '0') ? 0 : 1; }
    return g_conv_rows == 1;
}
}  // namespace delora

using namespace delora;

extern "C" int delora_conv_select_kernel(int rows_kernel) {
    const int prev = !use_conv_rows() ? 0 : (rows_use_pairs() ? 1 : 2);
    if (rows_kernel == 0 || rows_kernel == 1) { g_conv_rows = rows_kernel; rows_set_pairs(1); }
    if (rows_kernel == 2) { g_conv_rows = 1; rows_set_pairs(0); }          // row-block kernel, single CTAs only
    return prev;
}

extern "C" int delora_conv2d_fprop_bf16(const void* x, const void* w, const void* residual, const void* saved, void* y,
                                        int B, int Hin, int Win, int Cin, int Cout, int ksize, int stride_h,
                                        int stride_w, int act, void* stream) {
    DELORA_CHECK_ARG(x && w && y, "delora_conv2d_fprop_bf16: null pointer");
    DELORA_CHECK_ARG(act >= 0 && act <= 4 && (act < 3 || saved), "delora_conv2d_fprop_bf16: act=%d (3/4 need `saved`)", act);
    DELORA_CHECK_ARG(ksize == 3 || ksize == 1, "delora_conv2d_fprop_bf16: kernel size %d unsupported", ksize);
    DELORA_CHECK_ARG(Cin % 64 == 0 && Cout % 64 == 0, "delora_conv2d_fprop_bf16: Cin=%d, Cout=%d must be multiples of 64",
                     Cin, Cout);
    DELORA_CHECK_ARG((stride_h == 1 || stride_h == 2) && (stride_w == 1 || stride_w == 2) && Hin >= 1 && Win >= 1,
                     "delora_conv2d_fprop_bf16: stride (%d,%d) unsupported", stride_h, stride_w);
    if (stride_h == 1 && stride_w == 1 && conv_rows_eligible(Cin, Cout, ksize, Win) && use_conv_rows())
        return conv_rows_launch(x, w, residual, saved, y, B, Hin, Win, Cin, Cout, ksize, 1, 1, act, (cudaStream_t)stream, 0);
    ConvParams p;
    p.B = B; p.Cin = Cin; p.Cout = Cout; p.ksize = ksize; p.taps = ksize * ksize;
    p.stride_h = stride_h; p.stride_w = stride_w; p.pad_off = (ksize == 1) ? 1 : 0; p.act = act;
    // 3x3 / pad 1 and 1x1 / pad 0 both give floor((n - 1) / stride) + 1 outputs
    p.Hout = (Hin - 1) / stride_h + 1; p.Wout = (Win - 1) / stride_w + 1;
    pick_tile(p.Hout, p.Wout, kBlockM, &p.TW, &p.TH);
    p.tiles_w = (p.Wout + p.TW - 1) / p.TW;
    p.tiles_h = (p.Hout + p.TH - 1) / p.TH;
    p.BN = (Cout % 128 == 0) ? 128 : 64;
    // two CTAs per SM: one CTA's epilogue overlaps the other's main loop (ring = 3 stages of 32 KB for
    // BN = 128, 4 stages of 24 KB for BN = 64; TMEM: 2 x BN <= 512 columns)
    p.stages = (p.BN == 128) ? 3 : 4;
    const TensorMaps* maps = get_maps(x, w, B, Hin, Win, Cin, Cout, p);
    DELORA_CHECK_ARG(maps != nullptr, "delora_conv2d_fprop_bf16: cuTensorMapEncodeTiled failed or is unavailable");
    const size_t smem = (size_t)p.stages * (kBlockM * kBlockK * 2 + p.BN * kBlockK * 2) + (2 * kMaxStages + 1) * 8 + 16 + 1024;
    int dev = 0;
    cudaGetDevice(&dev);
    static bool attr_set[64] = {};                       // the opt-in is per device (one process may drive several)
    if (dev < 64 && !attr_set[dev]) {
        cudaError_t e = cudaFuncSetAttribute(conv_fprop_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 113 * 1024);
        DELORA_CHECK_ARG(e == cudaSuccess, "delora_conv2d_fprop_bf16: smem opt-in failed: %s", cudaGetErrorString(e));
        attr_set[dev] = true;
    }
    dim3 grid(B * p.tiles_h * p.tiles_w, Cout / p.BN);
    conv_fprop_tc_kernel<<<grid, kConvThreads, smem, (cudaStream_t)stream>>>(
        maps->x, maps->w, (const __nv_bfloat16*)residual, (const __nv_bfloat16*)saved, (__nv_bfloat16*)y, p);
    DELORA_CHECK_LAUNCH("conv_fprop_tc_kernel");
    return 0;
}

extern "C" int delora_conv_weight_prep_bf16(const float* w, int Cout, int Cin, int ksize, int Cin_pad, void* w_fwd,
                                            void* w_flip, void* stream) {
    DELORA_CHECK_ARG(w && w_fwd && Cout > 0 && Cin > 0 && Cin_pad >= Cin && (ksize == 1 || ksize == 3),
                     "delora_conv_weight_prep_bf16: bad argument");
    const size_t total = (size_t)Cout * ksize * ksize * Cin_pad + (w_flip ? (size_t)Cin * ksize * ksize * Cout : 0);
    weight_prep_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        w, Cout, Cin, ksize, Cin_pad, (__nv_bfloat16*)w_fwd, (__nv_bfloat16*)w_flip);
    DELORA_CHECK_LAUNCH("weight_prep_kernel");
    return 0;
}

extern "C" int delora_images_to_nhwc_bf16(const float* image_1, const float* image_2, int B, int H, int W, int Cpad,
                                          void* x, void* stream) {
    DELORA_CHECK_ARG(image_1 && image_2 && x && Cpad >= 8 && Cpad % 8 == 0, "delora_images_to_nhwc_bf16: bad argument");
    const size_t total = (size_t)B * (H + 2) * (W + 2) * (Cpad / 8);
    images_to_nhwc_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        image_1, image_2, B, H, W, Cpad, (__nv_bfloat16*)x);
    DELORA_CHECK_LAUNCH("images_to_nhwc_kernel");
    return 0;
}

extern "C" int delora_maxpool_w_nhwc_bf16(const void* x, int B, int H, int W, int C, void* y, void* stream) {
    DELORA_CHECK_ARG(x && y && W % 2 == 0 && C % 2 == 0, "delora_maxpool_w_nhwc_bf16: bad argument");
    const size_t total = (size_t)B * H * (W / 2) * (C / 2);
    maxpool_nhwc_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)x, B, H, W, C, (__nv_bfloat16*)y);
    DELORA_CHECK_LAUNCH("maxpool_nhwc_kernel");
    return 0;
}

// split-K slices: enough CTAs for ~2 waves of the 148 SMs, at most 64 and at most one per 64-pixel tile
static int wgrad_tap_group(int Cin, int ksize) {          // taps per CTA: N = 64 * nb * tg <= 256
    const int nb = (Cin >= 256) ? 4 : (Cin / 64);
    return ksize == 3 ? (4 / nb >= 3 ? 3 : (4 / nb >= 2 ? 2 : 1)) : 1;
}

static int wgrad_splits(int B, int Hout, int Wout, int Cin, int Cout, int ksize) {
    const int nb = (Cin >= 256) ? 4 : (Cin / 64);
    const int tg = wgrad_tap_group(Cin, ksize);
    const int base_ctas = ksize * ((ksize + tg - 1) / tg) * ((Cout + 127) / 128) * (Cin / (64 * nb));
    int splits = (2 * kNumSMs + base_ctas - 1) / base_ctas;
    splits = splits < 1 ? 1 : (splits > 64 ? 64 : splits);
    int tw = 64, th = 1;
    pick_tile(Hout, Wout, 64, &tw, &th);
    const int k_tiles = B * ((Hout + th - 1) / th) * ((Wout + tw - 1) / tw);
    return splits > k_tiles ? (k_tiles > 0 ? k_tiles : 1) : splits;
}

extern "C" int64_t delora_conv2d_wgrad_scratch_floats(int B, int Hout, int Wout, int Cin, int Cout, int ksize) {
    int64_t n = (int64_t)wgrad_splits(B, Hout, Wout, Cin, Cout, ksize) * ksize * ksize * Cout * Cin;
    if (wgrad2_eligible(Cin, Cout, ksize, 1, 1)) {           // either kernel may run (delora_conv_select_kernel)
        const int64_t n1 = wgrad2_scratch_floats(B, Hout, Wout, Cin, Cout, 1), n2 = wgrad2_scratch_floats(B, Hout, Wout, Cin, Cout, 2);
        n = n > n1 ? n : n1;
        n = n > n2 ? n : n2;
    }
    return n;
}

extern "C" int delora_conv2d_wgrad_bf16(const void* x, const void* dz, float* dw, float* scratch, int B, int Hin, int Win,
                                        int Cin, int Cin_true, int Cout, int ksize, int stride_h, int stride_w,
                                        void* stream) {
    DELORA_CHECK_ARG(x && dz && dw && scratch, "delora_conv2d_wgrad_bf16: null pointer");
    DELORA_CHECK_ARG(ksize == 3 || ksize == 1, "delora_conv2d_wgrad_bf16: kernel size %d unsupported", ksize);
    DELORA_CHECK_ARG(Cin % 64 == 0 && Cout % 64 == 0 && Cin_true >= 1 && Cin_true <= Cin,
                     "delora_conv2d_wgrad_bf16: Cin=%d, Cout=%d must be multiples of 64", Cin, Cout);
    DELORA_CHECK_ARG((stride_h == 1 || stride_h == 2) && (stride_w == 1 || stride_w == 2) && Hin >= 1 && Win >= 1,
                     "delora_conv2d_wgrad_bf16: stride (%d,%d) unsupported", stride_h, stride_w);
    if (use_conv_rows() && wgrad2_eligible(Cin, Cout, ksize, stride_h, stride_w))
        return wgrad2_launch(x, dz, dw, scratch, B, Hin, Win, Cin, Cin_true, Cout, stride_h, stride_w, (cudaStream_t)stream);
    WgradParams p;
    p.B = B; p.Cin = Cin; p.Cout = Cout; p.ksize = ksize; p.taps = ksize * ksize;
    p.stride_h = stride_h; p.stride_w = stride_w; p.pad_off = (ksize == 1) ? 1 : 0;
    p.Hout = (Hin - 1) / stride_h + 1; p.Wout = (Win - 1) / stride_w + 1;
    pick_tile(p.Hout, p.Wout, 64, &p.TW, &p.TH);
    p.tiles_per_row = (p.Wout + p.TW - 1) / p.TW;
    p.row_tiles = (p.Hout + p.TH - 1) / p.TH;
    p.k_tiles = B * p.row_tiles * p.tiles_per_row;
    p.nb = (Cin >= 256) ? 4 : (Cin / 64);                    // N tile = 64, 128 or 256 input channels
    p.ci_tiles = Cin / (64 * p.nb);
    p.a_blocks = (Cout >= 128) ? 2 : 1;
    const int co_tiles = (Cout + 127) / 128;
    p.splits = wgrad_splits(B, p.Hout, p.Wout, Cin, Cout, ksize);
    p.tg = wgrad_tap_group(Cin, ksize);
    p.groups_per_row = (ksize + p.tg - 1) / p.tg;
    p.stages = (p.nb * p.tg == 4) ? 3 : 4;
    PFN_cuTensorMapEncodeTiled_v12000 encode = get_encode();
    DELORA_CHECK_ARG(encode != nullptr, "delora_conv2d_wgrad_bf16: cuTensorMapEncodeTiled not available");
    CUtensorMap map_dz, map_x;
    {
        const int Hp = p.Hout + 2, Wp = p.Wout + 2;
        // extents stop at the last REAL pixel (padded index Wout / Hout): a ragged K tile then reads zeros from
        // TMA's out-of-bounds fill instead of the circular halo column, so it adds nothing to the sum
        cuuint64_t dims[4] = {(cuuint64_t)Cout, (cuuint64_t)(Wp - 1), (cuuint64_t)(Hp - 1), (cuuint64_t)B};
        cuuint64_t strides[3] = {(cuuint64_t)Cout * 2, (cuuint64_t)Wp * Cout * 2, (cuuint64_t)Hp * Wp * Cout * 2};
        cuuint32_t box[4] = {64, (cuuint32_t)p.TW, (cuuint32_t)p.TH, 1};
        cuuint32_t estr[4] = {1, 1, 1, 1};
        CUresult rc = encode(&map_dz, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(dz), dims, strides, box, estr,
                             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        DELORA_CHECK_ARG(rc == CUDA_SUCCESS, "delora_conv2d_wgrad_bf16: tensor map (dz) failed: %d", (int)rc);
    }
    {
        const int Hp = Hin + 2, Wp = Win + 2;
        cuuint64_t dims[4] = {(cuuint64_t)Cin, (cuuint64_t)Wp, (cuuint64_t)Hp, (cuuint64_t)B};
        cuuint64_t strides[3] = {(cuuint64_t)Cin * 2, (cuuint64_t)Wp * Cin * 2, (cuuint64_t)Hp * Wp * Cin * 2};
        cuuint32_t box[4] = {64, (cuuint32_t)(p.TW * stride_w), (cuuint32_t)(p.TH * stride_h), 1};
        cuuint32_t estr[4] = {1, (cuuint32_t)stride_w, (cuuint32_t)stride_h, 1};
        CUresult rc = encode(&map_x, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(x), dims, strides, box, estr,
                             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        DELORA_CHECK_ARG(rc == CUDA_SUCCESS, "delora_conv2d_wgrad_bf16: tensor map (x) failed: %d", (int)rc);
    }
    const size_t smem = (size_t)p.stages * (2 + p.nb * p.tg) * 8192 + (2 * kMaxStages + 1) * 8 + 16 + 1024;
    int dev = 0;
    cudaGetDevice(&dev);
    static bool attr_set[64] = {};
    if (dev < 64 && !attr_set[dev]) {
        cudaError_t e = cudaFuncSetAttribute(conv_wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        DELORA_CHECK_ARG(e == cudaSuccess, "delora_conv2d_wgrad_bf16: smem opt-in failed: %s", cudaGetErrorString(e));
        attr_set[dev] = true;
    }
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid(p.ksize * p.groups_per_row, co_tiles * p.ci_tiles, p.splits);
    conv_wgrad_tc_kernel<<<grid, kConvThreads, smem, st>>>(map_dz, map_x, scratch, p);
    DELORA_CHECK_LAUNCH("conv_wgrad_tc_kernel");
    const size_t total = (size_t)Cout * Cin_true * p.taps;
    wgrad_reduce_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(scratch, p.splits, p.taps, Cout, Cin, Cin_true, dw);
    DELORA_CHECK_LAUNCH("wgrad_reduce_kernel");
    return 0;
}

extern "C" int delora_zero_upsample_nhwc_bf16(const void* x, int B, int H, int W, int C, int sh, int sw, int Hout,
                                              int Wout, void* y, void* stream) {
    DELORA_CHECK_ARG(x && y && C % 8 == 0 && sh >= 1 && sw >= 1, "delora_zero_upsample_nhwc_bf16: bad argument");
    DELORA_CHECK_ARG((Hout - 1) / sh + 1 == H && (Wout - 1) / sw + 1 == W,
                     "delora_zero_upsample_nhwc_bf16: %dx%d is not the stride-(%d,%d) input size of a %dx%d output", Hout,
                     Wout, sh, sw, H, W);
    const size_t total = (size_t)B * (Hout + 2) * (Wout + 2) * (C / 8);
    zero_upsample_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)x, B, H, W, C, sh, sw, Hout, Wout, (__nv_bfloat16*)y);
    DELORA_CHECK_LAUNCH("zero_upsample_kernel");
    return 0;
}

extern "C" int delora_maxpool_w_idx_nhwc_bf16(const void* x, int B, int H, int W, int C, void* y, void* idx, int act,
                                              int x_f16, void* stream) {
    DELORA_CHECK_ARG(x && y && idx && W % 2 == 0 && C % 8 == 0 && act >= 0 && act <= 2,
                     "delora_maxpool_w_idx_nhwc_bf16: bad argument");
    const size_t total = (size_t)B * H * (W / 2) * (C / 8);
    maxpool_idx_nhwc_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)x, B, H, W, C, (__nv_bfloat16*)y, (uint8_t*)idx, act, x_f16 ? 1 : 0);
    DELORA_CHECK_LAUNCH("maxpool_idx_nhwc_kernel");
    return 0;
}

extern "C" int delora_maxpool_w_bwd_nhwc_bf16(const void* dy, const void* idx, const void* a, int B, int H, int W, int C,
                                              int act, void* dz, int a_f16, void* stream) {
    DELORA_CHECK_ARG(dy && idx && a && dz && W % 2 == 0 && C % 8 == 0, "delora_maxpool_w_bwd_nhwc_bf16: bad argument");
    if (C == 64 && W % kPoolTW == 0 && B <= 65535) {
        dim3 grid((unsigned)(W / kPoolTW), (unsigned)((H + kPoolTH - 1) / kPoolTH), (unsigned)B);
        maxpool_bwd_tile_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
            (const __nv_bfloat16*)dy, (const uint8_t*)idx, (const __nv_bfloat16*)a, B, H, W, act, (__nv_bfloat16*)dz,
            a_f16 ? 1 : 0);
        DELORA_CHECK_LAUNCH("maxpool_bwd_tile_kernel");
        return 0;
    }
    const size_t total = (size_t)B * H * W * (C / 8);
    maxpool_bwd_act_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)dy, (const uint8_t*)idx, (const __nv_bfloat16*)a, B, H, W, C, act, (__nv_bfloat16*)dz,
        a_f16 ? 1 : 0);
    DELORA_CHECK_LAUNCH("maxpool_bwd_act_kernel");
    return 0;
}

extern "C" int delora_avgpool_bwd_nhwc_bf16(const float* g, const void* a, int B, int H, int W, int C, int act, void* dz,
                                            void* stream) {
    DELORA_CHECK_ARG(g && a && dz && C % 8 == 0, "delora_avgpool_bwd_nhwc_bf16: bad argument");
    const size_t total = (size_t)B * H * W * (C / 8);
    avgpool_bwd_act_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        g, (const __nv_bfloat16*)a, B, H, W, C, act, (__nv_bfloat16*)dz);
    DELORA_CHECK_LAUNCH("avgpool_bwd_act_kernel");
    return 0;
}

extern "C" int delora_avgpool_nhwc_bf16(const void* x, int B, int H, int W, int C, float* y, void* stream) {
    DELORA_CHECK_ARG(x && y && B > 0 && B <= 65535 && H > 0 && W > 0 && C > 0 && C % 64 == 0,
                     "delora_avgpool_nhwc_bf16: bad argument (C must be a multiple of 64, got %d)", C);
    avgpool_nhwc_kernel<<<dim3((unsigned)(C / 64), (unsigned)B), 256, 0, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)x, H, W, C, y);
    DELORA_CHECK_LAUNCH("avgpool_nhwc_kernel");
    return 0;
}

extern "C" int delora_nhwc_to_nchw_f32(const void* x, int B, int H, int W, int C, float* y, void* stream) {
    DELORA_CHECK_ARG(x && y, "delora_nhwc_to_nchw_f32: null pointer");
    const size_t total = (size_t)B * C * H * W;
    nhwc_to_nchw_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)x, B, H, W, C, y);
    DELORA_CHECK_LAUNCH("nhwc_to_nchw_kernel");
    return 0;
}
