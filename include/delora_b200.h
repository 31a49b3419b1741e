/*
 * delora_b200 — C ABI of the B200-native (sm_100a) DeLORA hot path.
 *
 * The reference (leggedrobotics/delora) is pure Python with no FFI layer of its own; its
 * operator surface for this path is the set of Python methods cited on each entry point
 * below (paths relative to the reference root).  Every function here is what a ctypes
 * binding of that method calls; `delora_b200/_lib.py` is that binding and INTEGRATION.md
 * shows the stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (torch allocates), unless the
 *     parameter name starts with `h_`;
 *   - `stream` is a `cudaStream_t` passed as `void*` (NULL = legacy default stream); all
 *     work is enqueued on it and nothing synchronises the device;
 *   - return value: 0 = ok, non-zero = error; `delora_last_error()` returns a thread-local,
 *     NUL-terminated description of the last failure on the calling thread;
 *   - no global mutable state: scratch memory is passed in by the caller.  Functions are
 *     re-entrant per stream.
 *   - batches: `B` independent scans / scan pairs per call, one launch per operator for the
 *     whole batch.  Variable-length lists are padded to a stride with a device-side count.
 */
#ifndef DELORA_B200_H_
#define DELORA_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DELORA_B200_ABI_VERSION 1

/* float4-packed list element: (x, y, z, tag).  `tag` is an int32 bit pattern or a float flag,
 * as documented per array. */
typedef struct { float x, y, z, w; } delora_f4;

/* loss switches (config/hyperparameters.yaml:14-19) */
#define DELORA_LOSS_PO2PO        1u   /* point_to_point_loss                 */
#define DELORA_LOSS_PO2PL        2u   /* point_to_plane_loss                 */
#define DELORA_LOSS_PL2PL        4u   /* plane_to_plane_loss                 */
#define DELORA_NORMAL_LINEAR     8u   /* normal_loss: "linear" (default "squared") */
#define DELORA_ICP_STATS       256u  /* diagnostic: count the work of the NN search (delora_icp_stats) */

/* number of floats in one row of the `losses` output of delora_icp_fwd_bwd */
#define DELORA_LOSS_ROW 8   /* [po2po, po2pl, pl2pl, M_pairs, M_po2po, 0, 0, 0] */
/* number of floats per block-partial row in the icp workspace */
#define DELORA_ICP_PARTIAL 40

int         delora_abi_version(void);
const char* delora_last_error(void);

/* ---------------------------------------------------------------------------------------
 * Spherical projection.
 * Replaces utility.projection.ImageProjectionLayer.project_to_img
 *   (src/utility/projection.py:48-106; (u,v): :21-31; dedupe: :34-43).
 *
 * points     [B, C, n_stride] fp32 channels-first (x, y, z, extra channels...)
 * n_points   [B] int32 (device): valid points of each scan (<= n_stride)
 * keys       [B, H*W] uint64 scratch.  MUST be all-ones (0xFF bytes) on entry; it is all-ones
 *            again on exit (the resolve pass resets it), so one memset at allocation suffices.
 * image      [B, C+1, H, W] fp32 out: channels of the closest point per pixel + its range;
 *            empty pixels are 0.
 * index_map  [B, H, W] int32 out: index (into the scan) of the point kept in the pixel, -1 if empty.
 * hfov/vfov  radians, as the reference's bin scripts hand them over (bin/run_training.py:62-67).
 * div_mode   0: (a - f0) / span   (torch CPU op sequence, the golden vectors)
 *            1: (a - f0) * (1/span)  (torch CUDA's scalar-divide kernel) — see DESIGN.md.
 * Tie rule: equal fp32 range in one pixel -> lowest point index wins.
 */
int delora_project_fwd(const float* points, const int32_t* n_points, int B, int C, int n_stride,
                       int H, int W, double hfov0, double hfov1, double vfov0, double vfov1,
                       int div_mode, uint64_t* keys, float* image, int32_t* index_map, void* stream);

/* (u, v) of every point, un-rounded, in the ORIGINAL point order (the reference returns them
 * permuted by its range sort; see delora_sort_by_range).  src/utility/projection.py:21-31.
 * u, v: [B, n_stride] fp32 out; range: [B, n_stride] fp32 out (may be NULL). */
int delora_project_uv(const float* points, const int32_t* n_points, int B, int C, int n_stride,
                      int H, int W, double hfov0, double hfov1, double vfov0, double vfov1,
                      int div_mode, float* u, float* v, float* range, void* stream);

/* Stable ascending sort of each scan's points by fp32 range (ties: lower index first):
 * the order `torch.argsort(range)` imposes in src/utility/projection.py:63-67, made
 * deterministic.  LSD radix sort, 4 passes of 8 bits, one launch set for the batch.
 * range      [B, n_stride] fp32 (non-negative; NaN sorts last)
 * order      [B, n_stride] int32 out: point indices in ascending (range, index) order
 * scratch    bytes >= delora_sort_scratch_bytes(B, n_stride)
 */
int64_t delora_sort_scratch_bytes(int B, int n_stride);
int delora_sort_by_range(const float* range, const int32_t* n_points, int B, int n_stride,
                         int32_t* order, void* scratch, void* stream);

/* ---------------------------------------------------------------------------------------
 * Per-pixel normals.
 * Replaces preprocessing.normal_computation.NormalsComputer.compute_normal_vectors
 *   (src/preprocessing/normal_computation.py:89-122, :53-87) and utility.linalg.cov
 *   (src/utility/linalg.py:33-56).
 *
 * image      [B, C_img, H, W] fp32 (first three channels are x, y, z)
 * nb_h, nb_w neighbourhood side lengths (7, 11); patch = (2*(nb_h/2)+1) x (2*(nb_w/2)+1), edge-clamped
 * normals    [B, 3, H, W] fp32 out (may be NULL); 0 where the pixel is not valid (x!=0 & y!=0 & z!=0)
 *            or has fewer than `min_neighbors` range-gated neighbours.
 * pts_grid   [B, H*W] float4 out or NULL: (x, y, z, bits(pixel id)) of valid pixels, (+inf,+inf,+inf,-1) else
 * nrm_grid   [B, H*W] float4 out or NULL: (nx, ny, nz, has_normal ? 1 : 0)   (both or neither)
 *            -- the dense layout delora_icp_dense_fwd_bwd consumes (one point per spherical cell).
 */
int delora_normals_fwd(const float* image, int B, int C_img, int H, int W, int nb_h, int nb_w,
                       float epsilon_range, int min_neighbors, float* normals,
                       delora_f4* pts_grid, delora_f4* nrm_grid, void* stream);
/* How the 7x11 kernel stages its halo tile: 0 (default) coalesced loads + clamp + repack in one pass; 1 one TMA box
 * (cp.async.bulk.tensor.4d, three channel planes) + the same repack from shared memory (needs W % 4 == 0 and a 16-byte
 * aligned image, else mode 0 is used).  Results are bit-identical; mode 1 exists to measure what TMA buys this kernel
 * (DESIGN.md 4.2).  Returns the previous mode. */
int delora_normals_select_staging(int mode);

/* ---------------------------------------------------------------------------------------
 * Image -> lists (row-major order of the valid pixels), the layout the reference stores and
 * trains on (src/preprocessing/normal_computation.py:30-41, :84-87;
 * src/preprocessing/preprocesser.py:64-68), plus the cell index used by the NN search.
 *
 * pts4       [B, H*W] out: (x, y, z, bits(pixel id))    for the P_b valid pixels, in order
 * nrm4       [B, H*W] out: (nx, ny, nz, has_normal ? 1 : 0)
 * cell_start [B, H*W + 1] int32 out: exclusive prefix of the valid flags (CSR over pixels)
 * counts     [B] int32 out: P_b
 * scratch    int32 [B * delora_scan_blocks(H*W)]
 */
int delora_scan_blocks(int n_cells);
int delora_lists_from_images(const float* image, const float* normals, int B, int C_img, int H, int W,
                             delora_f4* pts4, delora_f4* nrm4, int32_t* cell_start, int32_t* counts,
                             int32_t* scratch, void* stream);

/* Bin arbitrary point lists (the reference's [1,3,N] tensors) into the spherical cell grid:
 * counting sort by cell.  Needed by losses.icp_losses.ICPLosses.forward for lists that did
 * not come from delora_lists_from_images (src/losses/icp_losses.py:34 builds a cKDTree here).
 * Points outside the field of view are clamped into the border cells (the search stays exact).
 *
 * pts, nrm   [B, 3, n_stride] fp32 channels-first;  n [B] int32
 * pts4/nrm4  [B, n_stride] out, sorted by cell; pts4.w = bits(original list index)
 * cell_start [B, H*W+1] int32 out
 * cursor     [B, H*W] int32 scratch (any contents), scratch int32 [B*delora_scan_blocks(H*W)]
 */
int delora_grid_build(const float* pts, const float* nrm, const int32_t* n, int B, int n_stride,
                      int H, int W, double hfov0, double hfov1, double vfov0, double vfov1,
                      delora_f4* pts4, delora_f4* nrm4, int32_t* cell_start, int32_t* cursor,
                      int32_t* scratch, void* stream);

/* Dense grids for the training step: the scan's points and its per-point (precomputed) normals,
 * gathered through the projection's pixel -> point index map (src/deploy/deployer.py:258-261).
 * points [B,C,n_stride], normal_lists [B,3,n_stride], index_map [B,H,W] ->
 * pts_grid/nrm_grid [B,H*W] float4 as delora_icp_dense_fwd_bwd expects them. */
int delora_grids_from_projection(const float* points, const float* normal_lists, const int32_t* index_map,
                                 int B, int C, int n_stride, int H, int W,
                                 delora_f4* pts_grid, delora_f4* nrm_grid, void* stream);

/* Pack channels-first lists to float4 (no sorting): pts4.w = bits(list index), nrm4.w = has_normal. */
int delora_pack_lists(const float* pts, const float* nrm, const int32_t* n, int B, int n_stride,
                      delora_f4* pts4, delora_f4* nrm4, void* stream);

/* ---------------------------------------------------------------------------------------
 * Fused SE(3) transform + exact nearest neighbour + ICP losses, forward and backward.
 * Replaces, per scan pair:
 *   deploy.deployer.Deployer.{transform,rotate}_point_cloud_transformation_matrix  (src/deploy/deployer.py:181-189)
 *   losses.icp_losses.ICPLosses.forward          (src/losses/icp_losses.py:28-158; cKDTree :34, query :24-26)
 *   KDPointToPlaneLoss / KDPlaneToPlaneLoss / KDPointToPointLoss   (:196-206, :224-240, :168-179)
 *   and autograd's backward of those down to the 3x4 transform (SURVEY.md §3.4).
 *
 * src_pts4/src_nrm4 [B, src_stride]: source points / normals BEFORE the transform (nrm4.w ignored;
 *                   has-normal is decided on the rotated normal as the reference does, :48-50)
 * n_src             [B] int32
 * T                 [B, 12] fp32 row-major 3x4 (R | t); NULL = identity (inputs already transformed)
 * tgt_pts4/tgt_nrm4 [B, tgt_stride] sorted by cell (from delora_lists_from_images / delora_grid_build)
 * cell_start        [B, H*W+1]
 * lambda_po2pl      weight of the po2pl term in the gradient (deployer.py:310)
 * flags             DELORA_LOSS_* bits
 * losses            [B, DELORA_LOSS_ROW] out (unweighted means, as ICPLosses returns them)
 * grad_T            [B, 12] out: d(po2po + lambda*po2pl + pl2pl)/d(R|t), row-major 3x4
 * nn_index          [B, src_stride] int32 out or NULL: tag (tgt_pts4.w bits) of the NN of every source point
 * point_dir         [B, src_stride] float4 out or NULL: unscaled d(loss)/d(source point): r*n_t with w = 1 for a
 *                   kept (normal, normal) pair; (s - t) with w = 2 for a po2po pair; w = 0 otherwise
 * normal_dir        [B, src_stride] float4 out or NULL: unscaled d(pl2pl)/d(source normal)
 *                   (delora_icp_point_grads turns the two into the reference-shaped gradients)
 * scratch           fp32 [delora_icp_scratch_floats(B, src_stride)]: per-warp partial rows, column sums and
 *                   B int32 completion counters (+ the dense path's range pyramid and work list).  Zero it ONCE after
 *                   allocation; every call leaves the counters at zero again.  The layout depends on (B, src_stride):
 *                   a buffer that is reused with a different batch size or image size must be zeroed again first.
 * The NN is the exact float64 Euclidean nearest neighbour (lowest tag on exact ties).
 */
int     delora_icp_partial_rows(int src_stride);
int64_t delora_icp_scratch_floats(int B, int src_stride);
int delora_icp_fwd_bwd(const delora_f4* src_pts4, const delora_f4* src_nrm4, const int32_t* n_src,
                       int src_stride, const float* T,
                       const delora_f4* tgt_pts4, const delora_f4* tgt_nrm4, const int32_t* cell_start,
                       int tgt_stride, int B, int H, int W,
                       double hfov0, double hfov1, double vfov0, double vfov1,
                       float lambda_po2pl, uint32_t flags,
                       float* losses, float* grad_T, int32_t* nn_index,
                       delora_f4* point_dir, delora_f4* normal_dir,
                       float* scratch, void* stream);

/* The same operator on dense range-image grids (the layout delora_normals_fwd writes): source =
 * the valid pixels of `src_grid`, target = `tgt_grid`, at most one point per cell, so neither
 * list compaction nor a CSR index is needed.  This is the training-step fast path
 * (src/deploy/deployer.py:252-261 keeps exactly one point per pixel of both scans).
 * src_grid/src_ngrid, tgt_grid/tgt_ngrid: [B, H*W] float4;  T: [B, 12];
 * scratch: fp32 [delora_icp_scratch_floats(B, H*W)], zeroed once (see above).
 * Launches block_range_kernel, icp_dense_kernel (window search, at most 16 growing steps per warp; the environment
 * variable DELORA_ICP_MAX_STRIPS overrides the limit for profiling), icp_dense_pending_kernel (range-pruned block
 * search of the lanes still open) and icp_finalize_kernel; results do not depend on the limit. */
int delora_icp_dense_fwd_bwd(const delora_f4* src_grid, const delora_f4* src_ngrid, const float* T,
                             const delora_f4* tgt_grid, const delora_f4* tgt_ngrid, int B, int H, int W,
                             double hfov0, double hfov1, double vfov0, double vfov1,
                             float lambda_po2pl, uint32_t flags, float* losses, float* grad_T,
                             float* scratch, void* stream);

/* Diagnostic for delora_icp_dense_fwd_bwd calls made with DELORA_ICP_STATS in `flags`: copies the 32 device
 * counters to the HOST array out32 (may be NULL) and optionally zeroes them.  [0] warps, [1] window-growing steps,
 * [2] cells evaluated per lane (both summed per warp), [3] warps that entered the range-pruned block search,
 * [4] lanes searched there, [5] blocks bounded, [6] blocks scanned, [7] max blocks scanned for one lane,
 * [8] float64 tie re-rankings, [9] max blocks bounded for one lane, [10] lanes with > 256 blocks, [11] lanes that
 * reached the block search without any candidate, [16..23] warps by number of steps {0, 1-2, 3-5, 6-10, 11-20, 21-40, 41-63, limit},
 * [24..31] cells per lane summed over the warps of the same bucket.  Synchronises the device. */
int delora_icp_stats(uint32_t* out32, int reset);

/* Backward of ICPLosses.forward w.r.t. its two differentiable inputs, for callers that hand in
 * already-transformed clouds and let autograd continue (src/deploy/deployer.py:294-307 -> :341):
 * upstream [B,3] = d(total)/d(loss_po2po, loss_po2pl, loss_pl2pl);  losses = the row written by
 * delora_icp_fwd_bwd;  grad_pts, grad_nrm: [B, 3, src_stride] channels-first out. */
int delora_icp_point_grads(const delora_f4* point_dir, const delora_f4* normal_dir, const int32_t* n_src,
                           int src_stride, int B, const float* losses, const float* upstream,
                           float* grad_pts, float* grad_nrm, void* stream);

/* ---------------------------------------------------------------------------------------
 * Encoder convolution, forward, on tcgen05 tensor cores (bf16 in, fp32 accumulate in TMEM, bf16 out).
 * Replaces the cuDNN call behind torch.nn.Conv2d in the reference's encoder
 *   (src/models/resnet_modified.py:40 stem, :126-134 conv3x3 / conv1x1; used at :95-120, :159-177)
 *   including the circular width padding (:97, :162, :167), the zero height padding, the
 *   activation and the residual add of BasicBlock.forward (:174-175).
 * x        [B, Hin+2, Win+2, Cin]  bf16 NHWC with materialised padding (rows 0/Hin+1 zero, column 0 =
 *          column Win, column Win+1 = column 1)
 * w        [Cout, ksize*ksize, Cin] bf16 (tap-major K: torch weight.permute(0,2,3,1))
 * residual [B, Hout+2, Wout+2, Cout] bf16 or NULL, added before the activation
 * y        [B, Hout+2, Wout+2, Cout] bf16 out (interior + circular halo columns are written; the
 *          zero halo rows must have been zeroed once by the caller)
 * saved    [B, Hout+2, Wout+2, Cout] bf16 or NULL: forward activation output for the backward modes
 * ksize 3 (pad 1 in H, wrap in W) or 1 (no padding); stride_h/w in {1,2};
 * act: 0 none, 1 relu, 2 tanh (forward);  3 / 4: multiply (acc + residual) by tanh'(saved) = 1 - saved^2 /
 *      relu'(saved) -- the data-gradient pass: dgrad of a stride-1 conv is this same kernel run on the output
 *      gradient with the flipped, transposed filter (strided convs: on the zero-upsampled gradient).
 * Cin, Cout multiples of 64 (the 8-channel stem input is channel-padded by delora_images_to_nhwc_bf16). */
int delora_conv2d_fprop_bf16(const void* x, const void* w, const void* residual, const void* saved, void* y, int B,
                             int Hin, int Win, int Cin, int Cout, int ksize, int stride_h, int stride_w, int act,
                             void* stream);
/* Measurement switch: 1 (default) lets delora_conv2d_fprop_bf16 use the row-block kernel (csrc/conv_rows.cu) for
 * stride-1 layers with Cout % 128 == 0, 0 keeps every layer on the tap-per-TMA kernel (csrc/conv_tc.cu); any other
 * value only queries.  2 keeps the row-block kernel but runs it on single CTAs only (no CTA pairs; same effect as
 * DELORA_CONV_PAIRS=0).  Returns the previous setting (0, 1 or 2).  0 has the same effect as the environment variable
 * DELORA_CONV_ROWS=0. */
int delora_conv_select_kernel(int rows_kernel);
/* Data gradient of a 3x3 convolution of stride (stride_h, stride_w) in {1,2}^2 -- autograd's backward of the same
 * nn.Conv2d layers (src/models/resnet_modified.py:126-134) w.r.t. their input -- by PHASE DECOMPOSITION: every
 * output phase (h % stride_h, w % stride_w) is a small convolution of the (un-upsampled) output gradient with the
 * subset of flipped taps that hits non-zero positions; no zero-upsampled tensor is materialised.
 * dz [B,Hout+2,Wout+2,Cout] (Hout = (Hin-1)/stride_h + 1 ...), w_flip [Cin, 9, Cout] (delora_conv_weight_prep_bf16),
 * residual / saved / dx [B,Hin+2,Win+2,Cin]; act as in delora_conv2d_fprop_bf16 (3 / 4 = multiply by act'(saved)).
 * residual_strided = 1: `residual` is [B,Hout+2,Wout+2,Cin] instead and is added at the input pixels
 * (stride_h * h, stride_w * w) only -- the data gradient of the block's 1x1 strided downsample (:134), which never
 * reaches the other pixels (replaces a zero-upsampled copy of it).
 * Needs Cout % 64 == 0, Cin % 128 == 0 (or Cin = 64 with >= 128 columns per phase and CTA pairs enabled) and, for stride_w = 2, an even Win (an odd circular width mixes the phases at
 * the seam: use delora_zero_upsample_nhwc_bf16 + delora_conv2d_fprop_bf16 there). */
int delora_conv2d_dgrad_bf16(const void* dz, const void* w_flip, const void* residual, const void* saved, void* dx,
                             int B, int Hin, int Win, int Cin, int Cout, int stride_h, int stride_w, int act,
                             int residual_strided, void* stream);
/* 1 if delora_conv2d_dgrad_bf16 takes this layer (forward Cin / Cout, input width, stride) under the current kernel
 * selection, else 0.  No GPU work; the answer changes with delora_conv_select_kernel(2) (Cin = 64 needs CTA pairs). */
int delora_conv2d_dgrad_supported(int Cin, int Cout, int Win, int stride_h, int stride_w);
/* Weight gradient of the same convolution on tcgen05 (split-K over pixels, deterministic reduction):
 * x [B,Hin+2,Win+2,Cin] padded NHWC bf16 (the layer input), dz [B,Hout+2,Wout+2,Cout] padded NHWC bf16
 * (gradient w.r.t. the pre-activation output) -> dw [Cout, Cin_true, k, k] fp32 (torch layout; Cin_true <= Cin
 * for the channel-padded stem).  scratch: fp32 [delora_conv2d_wgrad_scratch_floats(...)].
 * Any Hin, Win >= 1: Hout = (Hin-1)/stride_h + 1, Wout = (Win-1)/stride_w + 1; ragged tiles are zero-filled. */
int64_t delora_conv2d_wgrad_scratch_floats(int B, int Hout, int Wout, int Cin, int Cout, int ksize);
int delora_conv2d_wgrad_bf16(const void* x, const void* dz, float* dw, float* scratch, int B, int Hin, int Win,
                             int Cin, int Cin_true, int Cout, int ksize, int stride_h, int stride_w, void* stream);
/* y[h*sh, w*sw] = x[h, w], zero elsewhere (padded NHWC bf16 in and out): input of the dgrad of strided convs.
 * y is [B,Hout+2,Wout+2,C] with (Hout, Wout) the INPUT size of the strided convolution
 * ((Hout-1)/sh+1 == H, (Wout-1)/sw+1 == W: 45 -> 23 -> 45 for the odd widths of 64x720 images). */
int delora_zero_upsample_nhwc_bf16(const void* x, int B, int H, int W, int C, int sh, int sw, int Hout, int Wout,
                                   void* y, void* stream);

/* torch filter w [Cout,Cin,k,k] fp32 -> w_fwd [Cout,k*k,Cin_pad] bf16 (the `w` operand of delora_conv2d_fprop_bf16;
 * channels >= Cin zero) and, unless NULL, w_flip [Cin,k*k,Cout] bf16 (spatially flipped, in/out swapped: the filter
 * of the data-gradient pass).  One launch per layer and step replaces autograd's permute / flip / cast chain. */
int delora_conv_weight_prep_bf16(const float* w, int Cout, int Cin, int ksize, int Cin_pad, void* w_fwd, void* w_flip,
                                 void* stream);

/* All encoder filters in one launch (replaces 20 delora_conv_weight_prep_bf16 calls per training step).
 * table: device array of n_layers x 8 int64 = {fp32 weight ptr, w_fwd ptr, w_flip ptr or 0, Cout, Cin, k, Cin_pad, kind};
 * kind 0 = the layouts of delora_conv_weight_prep_bf16, kind 1 = the stem layout of delora_stem_weight_prep_bf16. */
int delora_conv_weight_prep_multi(const void* table, int n_layers, void* stream);

/* ---- Encoder stem (src/models/resnet_modified.py:40 conv1: 3x3, stride (1,2), 8 -> 64 channels, + activation :99) on a
 * 16-channel input layout; replaces the channel-padded (8 -> 64) route through delora_conv2d_fprop/wgrad_bf16.
 * x16    [B, H+2, W+2, 16] bf16: channels 0..7 = cat(image_1, image_2) (src/models/model.py:98), 8..15 zero, padding
 *        materialised as everywhere (delora_images_to_nhwc16_bf16 writes it)
 * w_stem [3, 64, 64] bf16: [filter row][output channel][k = q * 16 + c] (delora_stem_weight_prep_bf16)
 * y      [B, H+2, W/2+2, 64] bf16 out (fp16 bit patterns when out_f16 = 1);  dz same shape;  dw [64, Cin_true, 3, 3]
 *        fp32.  W must be even. */
int delora_images_to_nhwc16_bf16(const float* image_1, const float* image_2, int B, int H, int W, void* x16, void* stream);
int delora_stem_weight_prep_bf16(const float* w, int Cin, void* w_stem, void* stream);
int delora_stem_fprop_bf16(const void* x16, const void* w_stem, void* y, int B, int H, int W, int act, int out_f16,
                           void* stream);
int64_t delora_stem_wgrad_scratch_floats(int B, int H, int W);
int delora_stem_wgrad_bf16(const void* x16, const void* dz, float* dw, float* scratch, int B, int H, int W, int Cin_true,
                           void* stream);

/* cat(image_1, image_2) ([B,4,H,W] fp32 each, src/models/model.py:98) -> [B,H+2,W+2,Cpad] bf16 padded NHWC */
int delora_images_to_nhwc_bf16(const float* image_1, const float* image_2, int B, int H, int W, int Cpad,
                               void* x, void* stream);
/* MaxPool2d(3, stride (1,2), padding (1,0)) on the W-wrapped input (src/models/resnet_modified.py:46,:100-101) */
int delora_maxpool_w_nhwc_bf16(const void* x, int B, int H, int W, int C, void* y, void* stream);
/* training variants of the pools: forward with argmax (idx: uint8 [B,H,W/2,C]); backward of the max-pool
 * fused with act'(a) of the stem activation a; backward of the global average pool fused with act'(a) of
 * the last block (g: [B,C] fp32).  act: 0 none, 1 relu, 2 tanh.  All tensors padded NHWC bf16.
 * Pre-activation form (what the training path uses for the stem): the forward pool takes the stem's PRE-activation
 * z and applies `act` to the maximum (max act(z) = act(max z) for the monotonic tanh / relu); the backward then gets
 * `a` = z and act = 5 (relu'(z)) or 6 (tanh'(z) = 4 e^{-2|z|} / (1 + e^{-2|z|})^2): 1 - a^2 evaluated on a bf16-rounded,
 * saturated tanh output has no correct digit, the metre-valued inputs saturate the stem heavily.
 * x_f16 / a_f16 = 1: that tensor holds fp16 instead of bf16 values (delora_stem_fprop_bf16 with out_f16 = 1): three more
 * mantissa bits keep the pool's argmax on the fp32 winner when two window entries nearly tie. */
int delora_maxpool_w_idx_nhwc_bf16(const void* x, int B, int H, int W, int C, void* y, void* idx, int act, int x_f16,
                                   void* stream);
int delora_maxpool_w_bwd_nhwc_bf16(const void* dy, const void* idx, const void* a, int B, int H, int W, int C, int act,
                                   void* dz, int a_f16, void* stream);
int delora_avgpool_bwd_nhwc_bf16(const float* g, const void* a, int B, int H, int W, int C, int act, void* dz,
                                 void* stream);
/* AdaptiveAvgPool2d((1,1)) (src/models/resnet_modified.py:111): padded NHWC bf16 [B,H+2,W+2,C] -> y [B,C] fp32
 * (fp32 sums in a fixed order; C a multiple of 64) */
int delora_avgpool_nhwc_bf16(const void* x, int B, int H, int W, int C, float* y, void* stream);
/* padded NHWC bf16 -> NCHW fp32 (interior), the reference's feature-map layout */
int delora_nhwc_to_nchw_f32(const void* x, int B, int H, int W, int C, float* y, void* stream);

/* quaternion (x, y, z, w) + translation -> 4x4, and its backward.
 * Replaces models.model_parts.GeometryHandler.get_transformation_matrix_quaternion
 *   (src/models/model_parts.py:37-44 -> kornia 0.3.0 quaternion_to_rotation_matrix).
 * quaternion [B,4], translation [B,3] -> T [B,16].  grad variant: gT [B,16] -> gq [B,4], gt [B,3]. */
int delora_quat_to_T(const float* quaternion, const float* translation, int B, float* T, void* stream);
int delora_quat_to_T_bwd(const float* quaternion, const float* grad_T, int B,
                         float* grad_quaternion, float* grad_translation, void* stream);

/* ---- Data-parallel training step: average of the weight gradients over the ranks (SURVEY.md 8(e); the reference
 * steps one optimizer on one device, src/deploy/trainer.py:23-24, on `loss / batch_size`, src/deploy/deployer.py:329-342
 * -- equal per-rank batches + the mean over ranks reproduce it over the global batch).
 * One all-reduce of elements [offset, offset + count) of a flat fp32 buffer that is SYMMETRIC memory: allocated with
 * the same size on every rank of the node and mapped into every peer (CUDA VMM / torch symmetric memory).
 * peer_bufs[q] / peer_flags[q]: HOST arrays of `world` device addresses -- where rank q's flat buffer / flag words are
 *   mapped in THIS process (index `rank` = the local ones).  Flag words: delora_grad_allreduce_flag_words() uint32,
 *   zeroed once before the first call.
 * multicast_ptr: address of the flat buffer's NVSwitch multicast mapping, or 0 (then peers are read / written one by
 *   one in rank order).  seq: a counter that increases by one with every call, identical on all ranks.
 * scale: applied to the sum (1 / world for the average).  status: device int32, set non-zero if a peer did not arrive
 *   within 20 s (the kernel then carries on; it never hangs).  The kernel needs no shared memory and few registers so
 *   that its n_ctas CTAs are resident NEXT TO the persistent convolution CTAs and the reduction overlaps the backward.
 * n_ctas CTAs (<= 160) of n_threads threads (32 .. 128).
 * Every rank must call it with the same offset / count / seq / n_ctas / n_threads. */
int delora_grad_allreduce_flag_words(void);
int delora_grad_allreduce_f32(const uint64_t* peer_bufs, const uint64_t* peer_flags, uint64_t multicast_ptr, int rank,
                              int world, long long offset, long long count, float scale, uint32_t seq, int n_ctas,
                              int n_threads, int32_t* status, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DELORA_B200_H_ */
