// Encoder convolutions, second-generation kernel (round 2): row-block implicit GEMM with the filter taps issued from
// ONE halo tile in shared memory.
//
// Same operator as conv_tc.cu (the reference's nn.Conv2d layers, src/models/resnet_modified.py:126-134 used at
// :159-177; circular padding in W, zero padding in H, materialised in the padded NHWC bf16 layout) for the layers
// that carry the FLOPs: 3x3 (and 1x1) stride-1 convolutions with Cout % 128 == 0, and the data gradient of the
// strided 3x3 convolutions by PHASE DECOMPOSITION (each output phase (h % sh, w % sw) is a small convolution of the
// un-upsampled output gradient with a subset of the flipped taps: no zero-upsampled tensor, no MMAs on zeros).
//
// Why a second kernel: conv_tc.cu loads every (tap, 64-channel chunk) as its own TMA box, so an activation tile is
// fetched 9x from L2 and a 128 x 64 tile only buys 128 tensor cycles per 24 KB of shared-memory fill; profiles/
// r01_conv_tcgen05.md shows 4.0x DRAM over-read and 15-60 % tensor-pipe utilisation.  Here
//   * GEMM roles are swapped: M = 128 OUTPUT CHANNELS (A operand = filter tile [128 co][64 ci], K-major), N = the NS
//     pixels of one output-row segment (B operand = activation rows, K-major), so a job's accumulators are R rows x
//     NS pixels = <= 256 TMEM columns and ANY image width maps onto the N dimension (multiples of 16);
//   * per job and 64-channel chunk ONE TMA box brings the (R + 2) x (NS + 2) pixel halo tile; the B descriptor of
//     tap (r, q), row i starts at byte ((i + r) * (NS + 2) + q) * 128 of that tile -- the tensor core applies the
//     128-byte swizzle on absolute shared-memory addresses, so 128-byte-granular start offsets need no re-layout
//     (measured: scripts/umma_probe.cu, profiles/r02_umma_probe.log).  Activation traffic per MMA drops ~6x;
//   * CTAs are persistent (grid = min(jobs, SMs)), TMEM is allocated once (512 columns = two accumulator sets): the
//     epilogue of job j overlaps the MMAs of job j + 1; separate producer warps stream halo tiles (2 stages) and
//     filter tiles (4-6 stages);
//   * epilogue: tcgen05.ld gives a thread one channel x 32 pixels; a 32 x 32 transpose through shared memory turns
//     that into one pixel x 32 channels (64 contiguous bytes of NHWC), then residual / activation / act' / store as
//     in conv_tc.cu.
// Warp roles: 0 halo-tile producer, 1 filter producer, 2 MMA issuer + TMEM owner, 3..6 epilogue.
#include <string.h>
#include <stdlib.h>
#include "tc_common.cuh"

namespace delora {

constexpr int kRowsThreads = 224;                 // 3 role warps + 4 epilogue warps
constexpr int kRowsThreadsPixm = 352;             // pixel-on-M form: 8 epilogue warps (two per TMEM lane quarter; 156 regs/thread)
constexpr int kRowsMaxTaps = 9;
constexpr int kRowsMaxPhases = 4;
constexpr int kWTileBytes = 128 * 64 * 2;          // filter tile: 128 output channels x 64 input channels
// Dynamic shared memory of one persistent CTA: 226 KB, not the 227 KB maximum -- 228 KB per SM minus this and the 1 KB
// the system reserves per CTA leaves room for ONE more (shared-memory-free) CTA on the SM, which is what lets the
// gradient all-reduce kernel (grad_allreduce.cu) run beside the convolutions instead of between them.
constexpr int kRowsSmemBudget = 226 * 1024;

struct RowsPhase {
    int ntaps;
    int oh, ow;                                    // output pixel = (out_sh * h + oh, out_sw * w + ow)
    signed char drow[kRowsMaxTaps], dcol[kRowsMaxTaps], wtap[kRowsMaxTaps];
};

struct RowsParams {
    int B, Cin, Cout;
    int Hout, Wout;                                // output tensor (unpadded) size
    int Hg, Wg;                                    // job grid extent in phase coordinates (= Hout, Wout for stride 1)
    int out_sh, out_sw;
    int NS, R;                                     // pixels per row segment (MMA N), rows per job; R * NS <= 256
    int segs_w, blocks_h, co_tiles, kchunks;
    int n_phases;
    int n_jobs;
    int act;
    int w_stages;
    int a_stage_bytes;
    int n_tile;                                    // pixel-on-M mode: output channels per job (MMA N) = Cout <= 128
    int w_tile_bytes;                              // bytes of one filter tile in the ring
    int res_grid;                                  // 1: `residual` is given on the job grid [B, Hg+2, Wg+2, Cout] and belongs
                                                   //    to phase (0, 0) only (data gradient of a 1x1 strided downsample)
    RowsPhase phase[kRowsMaxPhases];
};

struct RowsJob { int ct, ph, b, h0, w0; };

// job -> (co tile, phase, image, first row, first column).  With CTA pairs (CG = 2) a job covers 2R rows (rank r takes
// rows h0 + r R .. + R - 1) and 256 output channels (rank r takes channels (2 ct + r) * 128 .. + 127).
__device__ __forceinline__ RowsJob rows_decode(const RowsParams& p, int job, int cg) {
    RowsJob j;
    j.ct = job % p.co_tiles; job /= p.co_tiles;
    j.w0 = (job % p.segs_w) * p.NS; job /= p.segs_w;
    j.h0 = (job % p.blocks_h) * p.R * cg; job /= p.blocks_h;
    j.b = job % p.B; job /= p.B;
    j.ph = job;                                    // phase-major: the phases with the most taps come first (host order)
    return j;
}

// CG = 1: one CTA per job, tcgen05.mma.cta_group::1 with M = 128 output channels, N = NS pixels.
// CG = 2: a CTA PAIR per job (cluster of 2, one per SM of a TPC), tcgen05.mma.cta_group::2 with M = 256 output
//         channels (128 per CTA: each CTA loads its own filter tile) and N = 2 NS pixels (each CTA loads the halo
//         tile of its own R rows): per SM the MMA reads 64 instead of 128 B/clk of shared memory and each filter
//         byte is fetched for twice the pixels -- measured necessary: the shared-memory port (128 B/clk, MMA operand
//         reads + TMA fills) is what bounds these kernels (scripts/umma_probe2.cu, profiles/r02_umma_probe2.log).
// PIXM (layers with Cout = 64 / 128, where M = 128 output channels cannot be filled): the roles are swapped back --
//         M = the 128 PIXELS of a row segment (A operand = halo-tile rows, same shifted descriptors), N = all Cout output
//         channels (B operand = filter tile [Cout / CG][64]); a thread of the epilogue owns a pixel, no transpose.
//         With CG = 2 the pair covers 2 x 128 pixels and each CTA loads half of the filter rows.
template <int CG, bool PIXM>
__global__ void __launch_bounds__(PIXM ? kRowsThreadsPixm : kRowsThreads, 1)
conv_rows_tc_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w,
                    const __nv_bfloat16* __restrict__ residual, const __nv_bfloat16* __restrict__ saved,
                    __nv_bfloat16* __restrict__ y, const __grid_constant__ RowsParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = DELORA_ALIGNED_SMEM(smem_raw);
    uint8_t* smem_a = smem;                                        // 2 halo-tile stages
    uint8_t* smem_w = smem_a + 2 * p.a_stage_bytes;                // filter ring
    float* stage = reinterpret_cast<float*>(smem_w + p.w_stages * p.w_tile_bytes);   // 4 x 4 KB transpose buffers
    uint64_t* a_full = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(stage) + 4 * 4096);
    uint64_t* a_empty = a_full + 2;
    uint64_t* acc_full = a_empty + 2;
    uint64_t* acc_empty = acc_full + 2;
    uint64_t* w_full = acc_empty + 2;
    uint64_t* w_empty = w_full + 8;
    uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(w_empty + 8);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int S = p.w_stages;
    const int pitch = p.NS + 2;                                    // pixels per halo-tile row
    const uint32_t rank = (CG == 2) ? cluster_ctarank() : 0u;
    const int unit = blockIdx.x / CG, n_units = gridDim.x / CG;    // CTA (pair) index / count

    if (threadIdx.x == 0) {
        for (int s = 0; s < 2; ++s) {
            mbar_init(a_full + s, 1); mbar_init(a_empty + s, 1);
            mbar_init(acc_full + s, 1); mbar_init(acc_empty + s, (PIXM ? 8 : 4) * CG);
        }
        for (int s = 0; s < S; ++s) { mbar_init(w_full + s, 1); mbar_init(w_empty + s, 1); }
        fence_barrier_init();
    }
    if (warp == 2) { if (CG == 2) tmem_alloc_2sm(tmem_ptr_smem, 512); else tmem_alloc(tmem_ptr_smem, 512); }
    tc_fence_before();
    __syncthreads();
    if (CG == 2) cluster_sync();                                   // peer barriers initialised before any remote arrive
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;

    if (warp == 0) {
        // ===================== halo-tile producer =====================
        if (lane == 0) {
            tma_prefetch_desc(&map_x);
            const uint32_t a_bytes = (uint32_t)(pitch * (p.R + 2) * 128);
            uint32_t it = 0;
            for (int job = unit; job < p.n_jobs; job += n_units) {
                const RowsJob j = rows_decode(p, job, CG);
                for (int kc = 0; kc < p.kchunks; ++kc, ++it) {
                    const uint32_t s = it & 1;
                    mbar_wait(a_empty + s, ((it >> 1) & 1) ^ 1);
                    // local (row j, pixel c) = padded input pixel (h0 + rank R + j, w0 + c)
                    if (CG == 2) {
                        if (rank == 0) mbar_expect_tx(a_full + s, 2 * a_bytes);
                        tma_load_4d_2sm(smem_a + s * p.a_stage_bytes, &map_x, a_full + s, kc * 64, j.w0,
                                        j.h0 + (int)rank * p.R, j.b);
                    } else {
                        mbar_expect_tx(a_full + s, a_bytes);
                        tma_load_4d(smem_a + s * p.a_stage_bytes, &map_x, a_full + s, kc * 64, j.w0, j.h0, j.b);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== filter producer =====================
        if (lane == 0) {
            tma_prefetch_desc(&map_w);
            uint32_t it = 0;
            for (int job = unit; job < p.n_jobs; job += n_units) {
                const RowsJob j = rows_decode(p, job, CG);
                const RowsPhase& ph = p.phase[j.ph];
                const int co0 = PIXM ? j.ct * p.n_tile + (int)rank * (p.n_tile / CG) : (j.ct * CG + (int)rank) * 128;
                const uint32_t wb = (uint32_t)p.w_tile_bytes;
                for (int kc = 0; kc < p.kchunks; ++kc)
                    for (int t = 0; t < ph.ntaps; ++t, ++it) {
                        const uint32_t s = it % S;
                        mbar_wait(w_empty + s, ((it / S) & 1) ^ 1);
                        if (CG == 2) {
                            if (rank == 0) mbar_expect_tx(w_full + s, 2 * wb);
                            tma_load_2d_2sm(smem_w + s * wb, &map_w, w_full + s, (int)ph.wtap[t] * p.Cin + kc * 64, co0);
                        } else {
                            mbar_expect_tx(w_full + s, wb);
                            tma_load_2d(smem_w + s * wb, &map_w, w_full + s, (int)ph.wtap[t] * p.Cin + kc * 64, co0);
                        }
                    }
            }
        }
    } else if (warp == 2) {
        // ===================== MMA issuer (leader CTA of a pair) =====================
        // The whole warp runs the loop (uniform control flow and operands -> uniform registers, no per-MMA
        // register -> uniform-register broadcasts); one elected lane issues the tcgen05 instructions.
        if (rank == 0) {
            const bool issuer = elect_one();
            const int N = PIXM ? p.n_tile : CG * p.NS, R = p.R, kchunks = p.kchunks;
            const uint32_t idesc = make_idesc(128 * CG, N, 0, 0);
            const uint64_t desc_hi = make_smem_desc(0);          // everything but the start-address field
            const uint32_t row_step = (uint32_t)(pitch * 128) >> 4;             // next tile row, in 16-byte units
            const uint32_t a_lo0 = (smem_u32(smem_a) & 0x3FFFFu) >> 4, a_step = (uint32_t)p.a_stage_bytes >> 4;
            const uint32_t w_lo0 = (smem_u32(smem_w) & 0x3FFFFu) >> 4;
            const int jobs_per_phase = p.co_tiles * p.segs_w * p.blocks_h * p.B;
            uint32_t as = 0, aph = 0, ws = 0, wph = 0, ab = 0, accph = 0;      // ring slots and phase bits
            int cur_phase = -1, ntaps = 0;
            uint32_t xoff[kRowsMaxTaps];                         // tap offsets inside the halo tile, 16-byte units
            for (int job = unit; job < p.n_jobs; job += n_units) {
                const int phase_id = job / jobs_per_phase;
                if (phase_id != cur_phase) {
                    cur_phase = phase_id;
                    const RowsPhase& ph = p.phase[phase_id];
                    ntaps = ph.ntaps;
#pragma unroll
                    for (int t = 0; t < kRowsMaxTaps; ++t) xoff[t] = (uint32_t)(((int)ph.drow[t] * pitch + (int)ph.dcol[t]) * 8);
                }
                mbar_wait(acc_empty + ab, accph ^ 1);            // epilogues drained this accumulator set
                tc_fence_after();
                const uint32_t acc = tmem_base + ab * 256;
                for (int kc = 0; kc < kchunks; ++kc) {
                    mbar_wait(a_full + as, aph);
                    tc_fence_after();
                    const uint32_t a_lo = a_lo0 + as * a_step;
#pragma unroll
                    for (int t = 0; t < kRowsMaxTaps; ++t) {
                        if (t < ntaps) {
                            mbar_wait(w_full + ws, wph);
                            tc_fence_after();
                            if (issuer) {
                                const uint64_t dw = desc_hi | (uint64_t)(w_lo0 + ws * ((uint32_t)p.w_tile_bytes >> 4));
                                const uint32_t x_lo = a_lo + xoff[t];
                                const uint32_t first = (kc == 0 && t == 0) ? 0u : 1u;
                                for (int i = 0; i < R; ++i) {
                                    const uint64_t dx = desc_hi | (uint64_t)(x_lo + (uint32_t)i * row_step);
#pragma unroll
                                    for (int k = 0; k < 4; ++k) {   // 64 channels = 4 x K16; +32 bytes = +2 in 16-byte units
                                        const uint64_t da = (PIXM ? dx : dw) + (uint64_t)(k * 2), db = (PIXM ? dw : dx) + (uint64_t)(k * 2);
                                        if (CG == 2)
                                            tcgen05_mma_bf16_2sm(acc + (uint32_t)(i * N), da, db, idesc, (k > 0) ? 1u : first);
                                        else
                                            tcgen05_mma_bf16(acc + (uint32_t)(i * N), da, db, idesc, (k > 0) ? 1u : first);
                                    }
                                }
                                if (CG == 2) tcgen05_commit_2sm(w_empty + ws); else tcgen05_commit(w_empty + ws);
                                if (t == ntaps - 1) {            // halo tile free after this chunk's last tap
                                    if (CG == 2) tcgen05_commit_2sm(a_empty + as); else tcgen05_commit(a_empty + as);
                                    if (kc == kchunks - 1) {     // accumulators of this job complete
                                        if (CG == 2) tcgen05_commit_2sm(acc_full + ab); else tcgen05_commit(acc_full + ab);
                                    }
                                }
                            }
                            __syncwarp();
                            if (++ws == (uint32_t)S) { ws = 0; wph ^= 1; }
                        }
                    }
                    as ^= 1; aph ^= (as == 0);
                }
                ab ^= 1; accph ^= (ab == 0);
            }
        }
    } else {
        // ===================== epilogue warps 3..6 =====================
        const int quarter = warp & 3;                            // TMEM lanes 32*quarter .. +31 = output channels
        float* st = stage + quarter * 1024;
        const int Wp = p.Wout + 2, Hp = p.Hout + 2;
        const int n_blocks = (CG * p.R * p.NS) >> 5;
        uint32_t j_it = 0;
        for (int job = unit; job < p.n_jobs; job += n_units, ++j_it) {
            const RowsJob j = rows_decode(p, job, CG);
            const RowsPhase& ph = p.phase[j.ph];
            const uint32_t ab = j_it & 1;
            // Both epilogue forms walk the job's 32-column accumulator blocks with the residual / saved loads of block
            // k + 1 in flight while block k is read from TMEM and stored (and block 0's loads issued before the
            // accumulators are even complete): the epilogue was stalled on exactly these global loads (ncu: the bf16
            // unpack after the residual load held 25 % of all samples, the tensor pipe idled behind acc_empty).
            struct Blk { size_t off, roff; bool in_range, use_res, hl, hr; };
            if (PIXM) {
                // lane = pixel of the segment, columns = output channels: no transpose
                const int wl = quarter * 32 + lane, wg = j.w0 + wl;
                const int wo = wg * p.out_sw + ph.ow;
                const int cpb = p.n_tile >> 5, nb = p.R * cpb;
                auto info = [&](int k) {
                    Blk bi;
                    const int i = k / cpb, c0 = (k - i * cpb) << 5;
                    const int hg = j.h0 + (int)rank * p.R + i;
                    const int ho = hg * p.out_sh + ph.oh;
                    bi.in_range = hg < p.Hg && wg < p.Wg && ho < p.Hout && wo < p.Wout;
                    bi.use_res = residual != nullptr && (!p.res_grid || (ph.oh | ph.ow) == 0);
                    const int c_first = j.ct * p.n_tile + c0;
                    bi.off = (((size_t)j.b * Hp + (ho + 1)) * Wp + (wo + 1)) * p.Cout + c_first;
                    bi.roff = p.res_grid ? (((size_t)j.b * (p.Hg + 2) + (hg + 1)) * (p.Wg + 2) + (wg + 1)) * p.Cout + c_first
                                         : bi.off;
                    bi.hr = wo == 0; bi.hl = wo == p.Wout - 1;
                    return bi;
                };
                const int ehalf = (warp - 3) >> 2;                // 0 / 1: which of the quarter's two warps
                Blk bn = info(ehalf < nb ? ehalf : 0);
                EpiloguePrefetch nxt;
                if (bn.in_range && ehalf < nb)
                    epilogue_prefetch32(nxt, bn.use_res ? residual + bn.roff : nullptr, saved + (p.act >= 3 ? bn.off : 0), 0, p.act);
                mbar_wait(acc_full + ab, (j_it >> 1) & 1);
                tc_fence_after();
                for (int k = ehalf; k < nb; k += 2) {             // the two warps of a lane quarter alternate blocks
                    const Blk bc = bn;
                    const EpiloguePrefetch cur = nxt;
                    if (k + 2 < nb) {
                        bn = info(k + 2);
                        if (bn.in_range)
                            epilogue_prefetch32(nxt, bn.use_res ? residual + bn.roff : nullptr, saved + (p.act >= 3 ? bn.off : 0), 0, p.act);
                    }
                    uint32_t acc[32];
                    tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + ab * 256 + (uint32_t)(k << 5), acc);
                    if (bc.in_range) {
                        float v[32];
#pragma unroll
                        for (int c = 0; c < 32; ++c) v[c] = __uint_as_float(acc[c]);
                        epilogue_finish32(v, cur, bc.use_res, y, bc.off, p.act, bc.hr, bc.hl, (size_t)p.Wout * p.Cout);
                    }
                }
            } else {
                const int c_first = (j.ct * CG + (int)rank) * 128 + quarter * 32;
                auto info = [&](int cb) {
                    // accumulator column -> (row i of the job, CTA half, pixel): columns of MMA i are [i][half][NS]
                    Blk bi;
                    const int col = cb * 32 + lane;
                    const int blk = col / p.NS, wl = col - blk * p.NS;
                    const int i = blk / CG, half = blk - i * CG;
                    const int hg = j.h0 + half * p.R + i, wg = j.w0 + wl;
                    const int ho = hg * p.out_sh + ph.oh, wo = wg * p.out_sw + ph.ow;
                    bi.in_range = hg < p.Hg && wg < p.Wg && ho < p.Hout && wo < p.Wout;
                    bi.use_res = residual != nullptr && (!p.res_grid || (ph.oh | ph.ow) == 0);
                    bi.off = (((size_t)j.b * Hp + (ho + 1)) * Wp + (wo + 1)) * p.Cout + c_first;
                    bi.roff = p.res_grid ? (((size_t)j.b * (p.Hg + 2) + (hg + 1)) * (p.Wg + 2) + (wg + 1)) * p.Cout + c_first
                                         : bi.off;
                    bi.hr = wo == 0; bi.hl = wo == p.Wout - 1;
                    return bi;
                };
                Blk bn = info(0);
                EpiloguePrefetch nxt;
                if (bn.in_range)
                    epilogue_prefetch32(nxt, bn.use_res ? residual + bn.roff : nullptr, saved + (p.act >= 3 ? bn.off : 0), 0, p.act);
                mbar_wait(acc_full + ab, (j_it >> 1) & 1);
                tc_fence_after();
                for (int cb = 0; cb < n_blocks; ++cb) {
                    const Blk bc = bn;
                    const EpiloguePrefetch cur = nxt;
                    if (cb + 1 < n_blocks) {
                        bn = info(cb + 1);
                        if (bn.in_range)
                            epilogue_prefetch32(nxt, bn.use_res ? residual + bn.roff : nullptr, saved + (p.act >= 3 ? bn.off : 0), 0, p.act);
                    }
                    uint32_t acc[32];
                    tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + ab * 256 + (uint32_t)(cb * 32), acc);
                    // transpose: thread = channel `lane` holds 32 pixels -> thread = pixel `lane` holds 32 channels.
                    // XOR-swizzled 32 x 32 fp32 tile: both directions are bank-conflict free
#pragma unroll
                    for (int jj = 0; jj < 32; ++jj) st[jj * 32 + (lane ^ jj)] = __uint_as_float(acc[jj]);
                    __syncwarp();
                    float v[32];
#pragma unroll
                    for (int c = 0; c < 32; ++c) v[c] = st[lane * 32 + (c ^ lane)];
                    __syncwarp();
                    if (bc.in_range)
                        epilogue_finish32(v, cur, bc.use_res, y, bc.off, p.act, bc.hr, bc.hl, (size_t)p.Wout * p.Cout);
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) { if (CG == 2) mbar_arrive_leader(acc_empty + ab); else mbar_arrive(acc_empty + ab); }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (CG == 2) cluster_sync();                                 // the peer may still be reading / signalling
    if (warp == 2) { if (CG == 2) tmem_dealloc_2sm(tmem_base, 512); else tmem_dealloc(tmem_base, 512); }
}

// ---------------------------------------------------------------- host side
static int rows_encode_maps(CUtensorMap* mx, CUtensorMap* mw, const void* x, const void* w, int B, int Hin, int Win,
                            int Cin, int Cout, int wtaps, int NS, int R, int w_rows) {
    PFN_cuTensorMapEncodeTiled_v12000 encode = get_tensor_map_encoder();
    if (!encode) return 1;
    const int Hp = Hin + 2, Wp = Win + 2;
    {
        cuuint64_t dims[4] = {(cuuint64_t)Cin, (cuuint64_t)Wp, (cuuint64_t)Hp, (cuuint64_t)B};
        cuuint64_t strides[3] = {(cuuint64_t)Cin * 2, (cuuint64_t)Wp * Cin * 2, (cuuint64_t)Hp * Wp * Cin * 2};
        cuuint32_t box[4] = {64, (cuuint32_t)(NS + 2), (cuuint32_t)(R + 2), 1};
        cuuint32_t estr[4] = {1, 1, 1, 1};
        if (encode(mx, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(x), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return 2;
    }
    {
        cuuint64_t dims[2] = {(cuuint64_t)wtaps * Cin, (cuuint64_t)Cout};
        cuuint64_t strides[1] = {(cuuint64_t)wtaps * Cin * 2};
        cuuint32_t box[2] = {64, (cuuint32_t)w_rows};
        cuuint32_t estr[2] = {1, 1};
        if (encode(mw, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(w), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return 3;
    }
    return 0;
}

// Tensor maps depend only on (pointers, shapes); the encoder's activations, filters and gradients live in
// persistent buffers, so a small per-thread cache removes the encode cost from the 40 launches of a step.
struct RowsMapKey { const void* x; const void* w; int B, Hin, Win, Cin, Cout, wtaps, NS, R, w_rows; };
struct RowsMapEntry { RowsMapKey k; CUtensorMap mx, mw; };

static const RowsMapEntry* rows_get_maps(const RowsMapKey& key) {
    static thread_local RowsMapEntry cache[128];
    static thread_local int used = 0, next = 0;
    for (int i = 0; i < used; ++i) {
        const RowsMapKey& c = cache[i].k;
        if (c.x == key.x && c.w == key.w && c.B == key.B && c.Hin == key.Hin && c.Win == key.Win && c.Cin == key.Cin &&
            c.Cout == key.Cout && c.wtaps == key.wtaps && c.NS == key.NS && c.R == key.R && c.w_rows == key.w_rows)
            return &cache[i];
    }
    RowsMapEntry& e = cache[next];
    if (rows_encode_maps(&e.mx, &e.mw, key.x, key.w, key.B, key.Hin, key.Win, key.Cin, key.Cout, key.wtaps, key.NS,
                         key.R, key.w_rows) != 0)
        return nullptr;
    e.k = key;
    const RowsMapEntry* out = &e;
    next = (next + 1) % 128;
    if (used < 128) ++used;
    return out;
}

// segment width / rows per job for a job grid of Hg x Wg positions: NS = multiple of 16 covering the row in equal
// segments of at most 128 pixels; R rows so that R * NS <= 256 accumulator columns (a multiple of 32)
static void rows_pick_tile(int Hg, int Wg, int cg, int* NS, int* R) {
    const int segs = (Wg + 127) / 128;
    int ns = ((Wg + segs - 1) / segs + 15) / 16 * 16;
    if (ns < 16) ns = 16;
    int r = 256 / (ns * cg);
    if (r < 1) r = 1;
    if (cg == 2) {                                  // columns per job = 2 R NS (a multiple of 32 for NS % 16 == 0)
        while (r > 1 && 2 * (r - 1) >= Hg) --r;     // no more rows than the image has
        *NS = ns; *R = r;
        return;
    }
    if ((r * ns) % 32 != 0) r -= 1;
    if (r > Hg) r = Hg;
    if (r < 1) r = 1;
    while ((r * ns) % 32 != 0) ++r;                 // r = 1 with ns % 32 == 16: take two rows (second one masked)
    *NS = ns; *R = r;
}

// DELORA_CONV_PAIRS=0 (or delora_conv_select_kernel(2)) keeps the single-CTA form for every layer
static int g_rows_pairs = -1;
bool rows_use_pairs() {
    if (g_rows_pairs < 0) { const char* e = getenv("DELORA_CONV_PAIRS"); g_rows_pairs = (e && e[0] == '0') ? 0 : 1; }
    return g_rows_pairs == 1;
}
void rows_set_pairs(int on) { g_rows_pairs = on ? 1 : 0; }

// pixel-on-M mode: Cout = 64 or 128 and a job grid at least one full 128-pixel segment wide
static bool rows_pixm(int Cout, int Wg) { return (Cout == 64 || Cout == 128) && Wg >= 128 && rows_use_pairs(); }

// Wg = width of the job grid (the output width for a stride-1 convolution, ceil(Wout / stride_w) for a data gradient)
bool conv_rows_eligible(int Cin, int Cout, int ksize, int Wg) {
    if (Cin % 64 != 0 || !(ksize == 3 || ksize == 1)) return false;
    return Cout % 128 == 0 || rows_pixm(Cout, Wg);
}

// stride-1 convolution (up_h = up_w = 1) or data gradient of a stride-(up_h, up_w) 3x3 convolution (x = output
// gradient of that convolution, w = its flipped / transposed filter [Cout][9][Cin], y = input gradient Hout x Wout)
int conv_rows_launch(const void* x, const void* w, const void* residual, const void* saved, void* y, int B, int Hout,
                     int Wout, int Cin, int Cout, int ksize, int up_h, int up_w, int act, cudaStream_t stream,
                     int residual_on_grid) {
    RowsParams p;
    memset(&p, 0, sizeof(p));
    p.res_grid = (residual_on_grid && (up_h > 1 || up_w > 1)) ? 1 : 0;
    p.B = B; p.Cin = Cin; p.Cout = Cout; p.Hout = Hout; p.Wout = Wout; p.act = act;
    p.out_sh = up_h; p.out_sw = up_w;
    p.Hg = (Hout + up_h - 1) / up_h; p.Wg = (Wout + up_w - 1) / up_w;
    const int Hin = (Hout - 1) / up_h + 1, Win = (Wout - 1) / up_w + 1;      // size of x (unpadded)
    if (ksize == 1) {
        p.n_phases = 1;
        p.phase[0].ntaps = 1; p.phase[0].drow[0] = 1; p.phase[0].dcol[0] = 1; p.phase[0].wtap[0] = 0;
    } else if (up_h == 1 && up_w == 1) {
        p.n_phases = 1;
        p.phase[0].ntaps = 9;
        for (int t = 0; t < 9; ++t) { p.phase[0].drow[t] = (signed char)(t / 3); p.phase[0].dcol[t] = (signed char)(t % 3); p.phase[0].wtap[t] = (signed char)t; }
    } else {
        // out[h][w] = sum_{r', q'} U[h + r' - 1][w + q' - 1] * Wf[r'][q'],  U = zero-upsampled x: only taps with
        // (h + r' - 1) % up_h == 0 and (w + q' - 1) % up_w == 0 contribute.  Phase (fh, fw): h = up_h * jh + fh.
        // Local halo-tile coordinates: padded x row jh0 + drow, drow = (fh + r' - 1) / up_h + 1 (same for columns).
        int np = 0;
        // phases ordered by decreasing tap count (static round-robin over CTAs: expensive jobs first)
        for (int pass = 9; pass >= 1; --pass)
            for (int fh = 0; fh < up_h; ++fh)
                for (int fw = 0; fw < up_w; ++fw) {
                    RowsPhase ph;
                    memset(&ph, 0, sizeof(ph));
                    ph.oh = fh; ph.ow = fw;
                    for (int r = 0; r < 3; ++r) {
                        if ((fh + r - 1 + up_h) % up_h != 0) continue;
                        for (int q = 0; q < 3; ++q) {
                            if ((fw + q - 1 + up_w) % up_w != 0) continue;
                            // floor division of (fh + r - 1) by up_h, values -1 .. 2
                            const int dr = (fh + r - 1 + up_h) / up_h - 1, dq = (fw + q - 1 + up_w) / up_w - 1;
                            ph.drow[ph.ntaps] = (signed char)(dr + 1); ph.dcol[ph.ntaps] = (signed char)(dq + 1);
                            ph.wtap[ph.ntaps] = (signed char)(r * 3 + q);
                            ++ph.ntaps;
                        }
                    }
                    if (ph.ntaps == pass) p.phase[np++] = ph;
                }
        p.n_phases = np;
    }
    const bool pixm = rows_pixm(Cout, p.Wg);
    const int cg = pixm ? (Cout == 128 ? 2 : 1) : ((Cout % 256 == 0 && rows_use_pairs()) ? 2 : 1);
    if (pixm) {
        p.NS = 128; p.R = (2 * cg <= p.Hg || cg == 1) ? 2 : 1;         // 128 pixels on M, R accumulators of Cout columns
        if (p.R > p.Hg) p.R = p.Hg;
        p.n_tile = Cout; p.w_tile_bytes = (Cout / cg) * 128;
        p.co_tiles = 1;
    } else {
        rows_pick_tile(p.Hg, p.Wg, cg, &p.NS, &p.R);
        p.n_tile = 0; p.w_tile_bytes = kWTileBytes;
        p.co_tiles = Cout / (128 * cg);
    }
    p.segs_w = (p.Wg + p.NS - 1) / p.NS;
    p.blocks_h = (p.Hg + p.R * cg - 1) / (p.R * cg);
    p.kchunks = Cin / 64;
    p.n_jobs = p.n_phases * B * p.blocks_h * p.segs_w * p.co_tiles;
    p.a_stage_bytes = (((p.NS + 2) * (p.R + 2) * 128) + 1023) / 1024 * 1024;
    const int fixed = 2 * p.a_stage_bytes + 4 * 4096 + 256 + 1024;
    int ws = (kRowsSmemBudget - fixed) / p.w_tile_bytes;
    if (ws > 8) ws = 8;
    DELORA_CHECK_ARG(ws >= 2, "conv_rows: tile %dx%d leaves no room for the filter ring", p.NS, p.R);
    p.w_stages = ws;
    const RowsMapKey key = {x, w, B, Hin, Win, Cin, Cout, ksize * ksize, p.NS, p.R, p.w_tile_bytes / 128};
    const RowsMapEntry* maps = rows_get_maps(key);
    DELORA_CHECK_ARG(maps != nullptr, "conv_rows: cuTensorMapEncodeTiled failed or is unavailable");
    const size_t smem = (size_t)fixed + (size_t)ws * p.w_tile_bytes;
    int dev = 0;
    cudaGetDevice(&dev);
    static bool attr_set[64] = {};
    if (dev < 64 && !attr_set[dev]) {
        cudaError_t e = cudaFuncSetAttribute(conv_rows_tc_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(conv_rows_tc_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(conv_rows_tc_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(conv_rows_tc_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        DELORA_CHECK_ARG(e == cudaSuccess, "conv_rows: shared-memory opt-in failed: %s", cudaGetErrorString(e));
        attr_set[dev] = true;
    }
    const int units = kNumSMs / cg;
    const int grid = (p.n_jobs < units ? p.n_jobs : units) * cg;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(pixm ? kRowsThreadsPixm : kRowsThreads);
    cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)cg; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    const __nv_bfloat16* res_p = (const __nv_bfloat16*)residual;
    const __nv_bfloat16* sav_p = (const __nv_bfloat16*)saved;
    __nv_bfloat16* y_p = (__nv_bfloat16*)y;
    cudaError_t le;
    if (pixm)
        le = (cg == 2) ? cudaLaunchKernelEx(&cfg, conv_rows_tc_kernel<2, true>, maps->mx, maps->mw, res_p, sav_p, y_p, p)
                       : cudaLaunchKernelEx(&cfg, conv_rows_tc_kernel<1, true>, maps->mx, maps->mw, res_p, sav_p, y_p, p);
    else
        le = (cg == 2) ? cudaLaunchKernelEx(&cfg, conv_rows_tc_kernel<2, false>, maps->mx, maps->mw, res_p, sav_p, y_p, p)
                       : cudaLaunchKernelEx(&cfg, conv_rows_tc_kernel<1, false>, maps->mx, maps->mw, res_p, sav_p, y_p, p);
    DELORA_CHECK_ARG(le == cudaSuccess, "conv_rows: launch failed: %s", cudaGetErrorString(le));
    DELORA_CHECK_LAUNCH("conv_rows_tc_kernel");
    return 0;
}

}  // namespace delora

using namespace delora;

// the shape conditions of delora_conv2d_dgrad_bf16 (forward Cin / Cout); they depend on the pair setting through
// rows_pixm, so callers ask here instead of restating them
extern "C" int delora_conv2d_dgrad_supported(int Cin, int Cout, int Win, int stride_h, int stride_w) {
    if (!((stride_h == 1 || stride_h == 2) && (stride_w == 1 || stride_w == 2) && Win >= 1)) return 0;
    if (stride_w == 2 && Win % 2 != 0) return 0;
    return conv_rows_eligible(Cout, Cin, 3, (Win + stride_w - 1) / stride_w) ? 1 : 0;
}

extern "C" int delora_conv2d_dgrad_bf16(const void* dz, const void* w_flip, const void* residual, const void* saved,
                                        void* dx, int B, int Hin, int Win, int Cin, int Cout, int stride_h, int stride_w,
                                        int act, int residual_strided, void* stream) {
    // Cin / Cout are those of the FORWARD convolution: dz has Cout channels, dx has Cin channels
    DELORA_CHECK_ARG(dz && w_flip && dx, "delora_conv2d_dgrad_bf16: null pointer");
    DELORA_CHECK_ARG(act >= 0 && act <= 4 && (act < 3 || saved), "delora_conv2d_dgrad_bf16: act=%d (3/4 need `saved`)", act);
    DELORA_CHECK_ARG((stride_h == 1 || stride_h == 2) && (stride_w == 1 || stride_w == 2) && Hin >= 1 && Win >= 1,
                     "delora_conv2d_dgrad_bf16: stride (%d,%d) unsupported", stride_h, stride_w);
    DELORA_CHECK_ARG(stride_w == 1 || Win % 2 == 0, "delora_conv2d_dgrad_bf16: stride_w = 2 needs an even Win (got %d)", Win);
    DELORA_CHECK_ARG(delora_conv2d_dgrad_supported(Cin, Cout, Win, stride_h, stride_w),
                     "delora_conv2d_dgrad_bf16: needs Cout %% 64 == 0 and Cin %% 128 == 0 (or Cin = 64 with at least "
                     "128 columns per phase and CTA pairs enabled); got Cin=%d, Cout=%d, Win=%d", Cin, Cout, Win);
    return conv_rows_launch(dz, w_flip, residual, saved, dx, B, Hin, Win, Cout, Cin, 3, stride_h, stride_w, act,
                            (cudaStream_t)stream, residual_strided);
}
