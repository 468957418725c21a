/*
 * t2h.h -- C ABI of the B200 (sm_100a) hot path of TomoSAR2Height.
 *
 * Every entry point replaces one third-party operator call of the reference
 * (paths relative to the reference repository).  The reference is pure Python, so the
 * "FFI" a maintainer binds is ctypes (see INTEGRATION.md); there are no torch types in
 * any signature: raw device pointers, sizes and a CUDA stream.
 *
 * Conventions
 *   - return value: 0 = ok, otherwise a T2H_ERR_* code (t2h_status_string() names it).
 *     Nothing throws across the boundary, nothing is allocated, freed or retained:
 *     the caller owns every buffer (inputs, outputs, workspaces).
 *   - all functions are re-entrant and hold no global or thread-local state (forward runs on
 *     the caller's thread, backward on the autograd thread); work is enqueued on `stream`.
 *   - "rows": per-point feature matrices are row-major (n_rows, C) fp32, one row per point.
 *   - "plane": feature planes are channels-last, (B, r, r, C) fp32, i.e. the memory layout of
 *     a torch (B, C, r, r) tensor with torch.channels_last strides.
 *   - "topology": points sorted by cell key.  key = b * R*R + code(ix, iy) with code = Morton
 *     (Z-order) interleave when `morton` != 0, else ix + R*iy.  With Morton keys the segments
 *     of every coarser power-of-two level r = R >> k are the key ranges
 *     [cell_start[s << 2k], cell_start[(s + 1) << 2k]), so ONE sort serves every level
 *     (`shift` = 2k below).  `perm[i]` is the row of the point at sorted position i; a NULL
 *     `perm` means rows are already stored in sorted order (the fused model path).
 *   - supported channel counts C: 4,8,16,32,64,128 and multiples of 128 up to 1024.
 */
#ifndef T2H_H_
#define T2H_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* t2h_stream_t; /* cudaStream_t */

enum {
  T2H_OK = 0,
  T2H_ERR_INVALID_ARGUMENT = 1,
  T2H_ERR_UNSUPPORTED_SHAPE = 2,
  T2H_ERR_CUDA = 3,
  T2H_ERR_WORKSPACE_TOO_SMALL = 4
};

int t2h_abi_version(void);
const char* t2h_status_string(int status);

/* ---- a1: utils/coordinate.py:12-28 coordinate2index --------------------------------------
 * out_index[i] = trunc(x*reso) + reso * trunc(y*reso), int64, no clamp (bit-exact). */
int t2h_cell_index(const float* xy, int64_t n_points, int64_t point_stride, int reso,
                   int64_t* out_index, t2h_stream_t stream);

/* ---- topology (replaces the 10-12 index recomputations per forward: pointnet.py:70,
 *      alto.py:80,190) ------------------------------------------------------------------- */
/* keys[i] = b*reso^2 + code(ix,iy) with (ix, iy) = trunc(x*reso), trunc(y*reso) as coordinate2index computes them;
 * b = i / n_per_batch.  The reference does not clamp (it relies on the crop of dataset.py:278 and fails in
 * torch_scatter otherwise): a point outside [0, 1)^2 (or NaN) is binned into the nearest border cell and
 * *range_flag (nullable device word) is set non-zero, so that the caller can raise like the reference would. */
int t2h_xy_keys(const float* xyz, int64_t n_points, int64_t point_stride, int64_t n_per_batch,
                int reso, int morton, int32_t* keys, int32_t* range_flag, t2h_stream_t stream);
/* ragged batches (tiles with different point counts, flat cloud + offsets[n_tiles + 1] on the device):
 * b = the tile whose range [offsets[b], offsets[b+1]) holds point i */
int t2h_xy_keys_ragged(const float* xyz, int64_t n_points, int64_t point_stride, const int64_t* offsets,
                       int n_tiles, int reso, int morton, int32_t* keys, int32_t* range_flag, t2h_stream_t stream);
/* keys[i] = b*dim_size + index[i]; *flag set non-zero if an index is outside [0, dim_size) */
int t2h_index_keys(const int64_t* index, int64_t n_points, int64_t n_per_batch, int64_t dim_size,
                   int32_t* keys, int32_t* flag, t2h_stream_t stream);
size_t t2h_sort_workspace_bytes(int64_t n_points);
/* stable sort by key (hand-written LSD radix sort, 8 bits per pass over the ceil(log2 n_keys) key bits: per-tile digit
 * histograms, per-digit scan, warp-ranked stable scatter); writes keys_sorted[n], perm[n] (sorted position -> input
 * position) and cell_start[n_keys + 1] (first sorted position of every key; cell_start[n_keys] = n; nullable) */
int t2h_sort_by_cell(const int32_t* keys, int64_t n_points, int64_t n_keys, void* workspace,
                     size_t workspace_bytes, int32_t* keys_sorted, int32_t* perm,
                     int32_t* cell_start, t2h_stream_t stream);
/* dst[i, :] = src[perm[i], :]  (rows of `width` floats; used for xyz and for re-ordering rows) */
int t2h_gather_rows(const float* src, const int32_t* perm, int64_t n_rows, int width, float* dst,
                    t2h_stream_t stream);
/* dst[perm[i], :] = src[i, :] */
int t2h_scatter_rows(const float* src, const int32_t* perm, int64_t n_rows, int width, float* dst,
                     t2h_stream_t stream);

/* ---- a2 / a3: segmented reductions over the sorted points ---------------------------------------
 * All of them are ROW-BALANCED: work is split into fixed chunks of consecutive sorted positions
 * (`row_keys[i]` = sort key of sorted position i, i.e. keys_sorted of t2h_sort_by_cell; the segment of a
 * level is row_keys[i] >> shift), so a cell with thousands of points costs the same per row as a cell with
 * one.  Cells inside a chunk are finished by the walker; cells that cross a chunk border leave partials in
 * `workspace` (t2h_seg_workspace_bytes) that a fix-up launch adds in chunk order.  No atomics.           */
size_t t2h_seg_workspace_bytes(int64_t n_rows, int64_t n_seg, int C);

/* a2: pointnet.py:92-99 pool_local = torch_scatter.scatter_max + gather.
 * Per segment and channel: max over the segment's rows, ties -> first row in sorted order
 * (= smallest point index, the torch_scatter CPU rule), empty -> 0 / arg -1.
 *   pooled (n_rows, C), nullable: the max broadcast back to every row of the segment (needs plane)
 *   plane  (n_seg, C),  nullable: the per-cell max, rows in row-major (b, y, x) cell order
 *   arg    (n_seg, C)  int32   : winning ROW index (same row order as plane), -1 if empty
 *   tie_rank, nullable: original point index of every sorted position; needed for the tie rule
 *     when a segment spans several sort keys (shift > 0), where sorted order != point order       */
int t2h_seg_max_fwd(const float* rows, int64_t n_rows, const int32_t* perm, const int32_t* tie_rank,
                    const int32_t* row_keys, const int32_t* cell_start, int64_t n_seg, int shift, int C,
                    int morton, int reso, void* workspace, size_t workspace_bytes, float* pooled,
                    float* plane, int32_t* arg, t2h_stream_t stream);
/* grad_rows[row, c] = (row == arg[seg, c]) ? sum_{rows of seg} grad_pooled[., c] + grad_plane[seg, c] : 0
 * (either gradient may be NULL; the workspace is only needed with grad_pooled) */
int t2h_seg_max_bwd(const float* grad_pooled, const float* grad_plane, int64_t n_rows, const int32_t* perm,
                    const int32_t* row_keys, const int32_t* cell_start, int64_t n_seg, int shift, int C,
                    int morton, int reso, const int32_t* arg, void* workspace, size_t workspace_bytes,
                    float* grad_rows, t2h_stream_t stream);

/* a3: pointnet.py:101-111, alto.py:76-88,187-197 torch_scatter.scatter_mean.
 * plane[cell, :] = sum of the segment's rows (/ count when mean != 0); empty cell -> 0.        */
int t2h_seg_reduce_fwd(const float* rows, int64_t n_rows, const int32_t* perm, const int32_t* row_keys,
                       const int32_t* cell_start, int64_t n_seg, int shift, int C, int morton, int reso,
                       int mean, void* workspace, size_t workspace_bytes, float* plane, t2h_stream_t stream);
/* rows[row, :] = plane[cell(row), :] (/ count when mean != 0): backward of the mean, and the
 * gather-back of pool_local when scatter_type == 'mean'; a pure row-parallel map               */
int t2h_seg_broadcast(const float* plane, int64_t n_rows, const int32_t* perm, const int32_t* row_keys,
                      const int32_t* cell_start, int64_t n_seg, int shift, int C, int morton, int reso,
                      int mean, float* rows, t2h_stream_t stream);
/* rows[row, :] = plane[cell(row), :] (/ count) + add_rows[row, :], and *absmax_slot (nullable) = bit pattern of max |rows|:
 * the backward of the mean-scatter fused with the accumulation of the OTHER gradient branch of the same per-point
 * tensor (alto.py:123-130: `c` feeds generate_plane_features and the next level's fc_c), so that autograd's add pass
 * and the operand-maximum pass of the GEMMs that consume the sum disappear */
int t2h_seg_broadcast_add(const float* plane, const float* add_rows, int64_t n_rows, const int32_t* perm,
                          const int32_t* row_keys, const int32_t* cell_start, int64_t n_seg, int shift, int C,
                          int morton, int reso, int mean, float* rows, uint32_t* absmax_slot, t2h_stream_t stream);
/* the scatter_mean pair under the names of SURVEY.md §8(b): = t2h_seg_reduce_fwd(mean = 1) / t2h_seg_broadcast(mean = 1) */
int t2h_seg_mean_fwd(const float* rows, int64_t n_rows, const int32_t* perm, const int32_t* row_keys,
                     const int32_t* cell_start, int64_t n_seg, int shift, int C, int morton, int reso,
                     void* workspace, size_t workspace_bytes, float* plane, t2h_stream_t stream);
int t2h_seg_mean_bwd(const float* grad_plane, int64_t n_rows, const int32_t* perm, const int32_t* row_keys,
                     const int32_t* cell_start, int64_t n_seg, int shift, int C, int morton, int reso,
                     float* grad_rows, t2h_stream_t stream);

/* ---- a4: alto.py:90-95,199-205 F.grid_sample(bilinear, border, align_corners=True) -----------
 * out_rows[row, :] = 4-tap bilinear sample of plane[b] at (x, y) = xyz_sorted[i, 0:2]
 * (point_stride, in floats, must be even: coordinates are fetched as one 8-byte load);
 * the tile of sorted point i is tile_ids[i] when given (ragged batches), else row / n_per_batch */
int t2h_bilinear_sample_fwd(const float* plane, int reso, int C, const float* xyz_sorted,
                            int64_t point_stride, const int32_t* perm, const int32_t* tile_ids,
                            int64_t n_points, int64_t n_per_batch, float* out_rows, t2h_stream_t stream);
/* grad_plane (B, r, r, C), atomic-free and deterministic (replaces grid_sampler_2d_backward's atomicAdd).
 * With Morton keys, `row_keys` and a workspace:
 *   - few rows per cell, C in {32, 64, 128}: warp-private shared-memory accumulator tiles over Morton blocks of
 *     cells with a one-cell halo (single writer per accumulator, sorted point order), region tiles merged in a
 *     fixed order;
 *   - otherwise (C = 32, 64 or a multiple of 128): row-balanced walk that keeps the nine (3x3 target) partial
 *     sums of the current cell in registers, chunk-border partials added in chunk order, then a 9-tap gather.
 * Else (workspace / row_keys NULL, row-major keys, other C): gather over the 3x3 neighbour cells of every
 * plane cell. */
size_t t2h_bilinear_sample_bwd_workspace_bytes(int reso, int C, int64_t n_points, int64_t n_seg, int morton);
int t2h_bilinear_sample_bwd(const float* grad_rows, int64_t n_points, int reso, int C,
                            const float* xyz_sorted, int64_t point_stride, const int32_t* perm,
                            const int32_t* row_keys, const int32_t* cell_start, int64_t n_seg, int shift,
                            int morton, void* workspace, size_t workspace_bytes, float* grad_plane,
                            t2h_stream_t stream);

/* ---- a5: pixel.py:105-111 F.interpolate(bilinear, align_corners=True) ----------------------- */
int t2h_upsample_bilinear_fwd(const float* in, int B, int h, int w, int C, int out_h, int out_w,
                              float* out, t2h_stream_t stream);
int t2h_upsample_bilinear_bwd(const float* grad_out, int B, int h, int w, int C, int out_h,
                              int out_w, float* grad_in, t2h_stream_t stream);

/* ---- a6-a9: nn.Linear on the point path (block/resnet.py:46-54, pointnet.py:36-40,72-82,
 *      alto.py:63-69,123-128,164-170,248-253, pixel.py:48-58) ------------------------------------
 * 3xTF32 on tcgen05 tensor cores (fp32 in/out, fp32-grade accuracy, fp32 accumulation in TMEM).
 *   out[r, n] = sum_k act(x[r, k]) * w[n, k] + bias[n]   (zeroed where mask[r, n] <= 0)   + residual[r, n]
 * x may be the concatenation [x1 | x2] along k (the torch.cat of pointnet.py:78) without materialising
 * it; act = ReLU when relu_in != 0.  The weight is passed pre-split (t2h_split_tf32) as w_hi / w_lo,
 * row-major [n_out, k1 + k2].  The same entry point serves the input-gradient GEMM of the backward
 * (x = grad_out, w = weight^T, mask = saved pre-activation, residual = gradient accumulated so far). */
int t2h_split_tf32(const float* w, int64_t n, float* hi, float* lo, t2h_stream_t stream);
int t2h_linear_fwd(const float* x1, int64_t ld_x1, int k1, const float* x2, int64_t ld_x2, int k2,
                   int64_t rows, const float* w_hi, const float* w_lo, int n_out, const float* bias,
                   int relu_in, const float* mask, int64_t ld_mask, const float* residual,
                   int64_t ld_res, float* out, int64_t ld_out, t2h_stream_t stream);

/* 3xFP16 flavour of the same GEMM for wide layers (n_out > 64): kind::f16 tensor-core passes run at twice
 * the TF32 rate.  Both operands are scaled by a power of two taken from their maximum magnitude (scaled
 * maximum in [2^14, 2^15), exact), split into fp16 hi = rn(v), lo = rn(v - hi), multiplied as
 * lo*hi + hi*lo + hi*hi with fp32 accumulation and un-scaled in the epilogue: 2^-22 relative per product,
 * plus an absolute floor of 2^-40 of the operand maximum for entries that are tiny against it.
 *   t2h_absmax:     *slot = bit pattern of max |[x1 | x2]| (x2 nullable / k2 = 0), pre-activation
 *   t2h_split_f16:  w (n fp32 values, n even) -> fp16 hi / lo under the scale of *absmax
 *   t2h_linear_fwd_f16: as t2h_linear_fwd with the fp16 weight split, (k1 + k2) % 8 == 0; out_absmax
 *                   (nullable) receives max |out|, i.e. the x_absmax of a following layer, for free */
int t2h_absmax(const float* x1, int64_t ld_x1, int k1, const float* x2, int64_t ld_x2, int k2,
               int64_t rows, uint32_t* slot, t2h_stream_t stream);
int t2h_split_f16(const float* w, int64_t n, const uint32_t* absmax, uint16_t* hi, uint16_t* lo,
                  t2h_stream_t stream);
/* out = a + b (n fp32 values, n % 4 == 0) and *slot = bit pattern of max |out|: the sum of the two gradient
 * branches of a tensor that is used twice (autograd's accumulation), with the operand maximum of the GEMM
 * that consumes it taken on the way */
int t2h_add_absmax(const float* a, const float* b, int64_t n, float* out, uint32_t* slot,
                   t2h_stream_t stream);
int t2h_linear_fwd_f16(const float* x1, int64_t ld_x1, int k1, const float* x2, int64_t ld_x2, int k2,
                       int64_t rows, const uint32_t* x_absmax, const uint16_t* w_hi,
                       const uint16_t* w_lo, const uint32_t* w_absmax, int n_out, const float* bias,
                       int relu_in, const float* mask, int64_t ld_mask, const float* residual,
                       int64_t ld_res, float* out, int64_t ld_out, uint32_t* out_absmax,
                       t2h_stream_t stream);

/* weight gradient grad_w[n, k] = sum_r grad_out[r, n] * act(x[r, k]) and (grad_b nullable) bias gradient
 * grad_b[n] = sum_r grad_out[r, n] (autograd backward of nn.Linear): 3xTF32 tcgen05 GEMM over
 * MN-major operands (grad_out^T through tensor memory), split over the rows, partials summed in a
 * fixed order */
size_t t2h_linear_wgrad_workspace_bytes(int64_t rows, int n_out, int k_in);
int t2h_linear_wgrad(const float* grad_out, int64_t ld_g, const float* x, int64_t ld_x, int64_t rows,
                     int n_out, int k_in, int relu_in, void* workspace, size_t workspace_bytes,
                     float* grad_w, int64_t ld_w, float* grad_b, t2h_stream_t stream);
/* 3xFP16 flavour of the weight gradient for k_in > 64: g^T as packed fp16 pairs through tensor memory, x
 * converted in shared memory to MN-major fp16 hi / lo tiles; operand scales from the two maxima (t2h_absmax).
 * Same workspace, split and reduction as t2h_linear_wgrad. */
int t2h_linear_wgrad_f16(const float* grad_out, int64_t ld_g, const uint32_t* g_absmax, const float* x,
                         int64_t ld_x, const uint32_t* x_absmax, int64_t rows, int n_out, int k_in,
                         int relu_in, void* workspace, size_t workspace_bytes, float* grad_w,
                         int64_t ld_w, float* grad_b, t2h_stream_t stream);
/* ---- f3 (SURVEY §8f): 3x3 / padding 1 convolutions of the plane CNN (alto.py:59-61,98-99,177-182,226-227,
 *      pixel.py:20-22) as implicit GEMM on the same tcgen05 3xTF32 pipeline.  Planes are channels-last
 *      (B, H, W, C); the weight is passed as the matrix [cout, 9*cin] with k = (3*ky + kx)*cin + ci
 *      (= the conv weight in torch.channels_last memory order), pre-split like a linear weight.
 *      out = conv3x3(act(x)) + bias  (zeroed where mask <= 0)  (+ residual); the input gradient is the
 *      same call with the spatially flipped, transposed weight.  Needs cin % 32 == 0, W % 16 == 0,
 *      H % 8 == 0 (forward) / H % 2 == 0 (weight gradient). */
int t2h_conv3x3_fwd(const float* x, int B, int H, int W, int cin, const float* w_hi, const float* w_lo,
                    int cout, const float* bias, int relu_in, const float* mask, const float* residual,
                    float* out, t2h_stream_t stream);
size_t t2h_conv3x3_wgrad_workspace_bytes(int B, int H, int W, int cin, int cout);
int t2h_conv3x3_wgrad(const float* grad_out, const float* x, int B, int H, int W, int cin, int cout,
                      int relu_in, void* workspace, size_t workspace_bytes, float* grad_w, float* grad_b,
                      t2h_stream_t stream);
/* 3xFP16 flavours of the two convolution GEMMs (operand scales as for t2h_linear_fwd_f16; the weight matrix
 * [cout, 9*cin] is split with t2h_split_f16). */
int t2h_conv3x3_fwd_f16(const float* x, int B, int H, int W, int cin, const uint32_t* x_absmax,
                        const uint16_t* w_hi, const uint16_t* w_lo, const uint32_t* w_absmax, int cout,
                        const float* bias, int relu_in, const float* mask, const float* residual,
                        float* out, uint32_t* out_absmax, t2h_stream_t stream);
int t2h_conv3x3_wgrad_f16(const float* grad_out, const uint32_t* g_absmax, const float* x,
                          const uint32_t* x_absmax, int B, int H, int W, int cin, int cout, int relu_in,
                          void* workspace, size_t workspace_bytes, float* grad_w, float* grad_b,
                          t2h_stream_t stream);
/* ---- f2 (SURVEY §8f): scene inference either side of the forward.  dataset.py:234,243-278 + utils/crop_cloud.py:21-29
 *      (strict 2-D crop, normalisation with the local z minimum, float cast, re-crop) and generator.py:139-154
 *      (flip, blend window, accumulation into the float64 scene rasters).
 * `points`: the scene cloud (n, 3) float64, binned by stride-sized cells so that a tile's candidates are a few
 * contiguous row ranges; `items`: work items of <= 1024 candidates, 16 bytes each {int32 tile, int32 count,
 * int64 first_row}; `tile_xy` (n_tiles, 2) float64 tile anchors (lower-left corner).
 *   t2h_tile_count: item_count[i] = survivors of both crops; tile_zmin[t] = order-preserving code of min z over the
 *                   first-crop survivors (initialise to all ones; an integer atomicMin, deterministic)
 *   t2h_tile_write: survivors as (x, y, z, 0) float32 rows in candidate order, item i starting at item_offset[i]
 *   t2h_blend_accumulate: for every raster pixel of the batch's bounding box, in tile order:
 *                   dsm += (double) heights[b, S-1-i, j] * wx[j] * wy[i];  weight += wx[j] * wy[i]            */
int t2h_tile_count(const double* points, const void* items, int64_t n_items, const double* tile_xy, double patch,
                   int32_t* item_count, uint64_t* tile_zmin, t2h_stream_t stream);
int t2h_tile_write(const double* points, const void* items, int64_t n_items, const double* tile_xy, double patch,
                   double z_scale, const int64_t* item_offset, const uint64_t* tile_zmin, float* out_xyz0,
                   t2h_stream_t stream);
int t2h_blend_accumulate(const float* heights, int n_tiles, int S, const int32_t* t_row, const int32_t* l_col,
                         const double* wx, const double* wy, int r0, int c0, int box_rows, int box_cols, int n_rows,
                         int n_cols, double* dsm, double* weight, t2h_stream_t stream);
/* orthophoto windows of a tile batch (models with the image branch, model.py:54-67), cut from a planar float32 scene
 * raster (C, rows, cols) that stays on the device:
 *   out[b, h, j, c] = (raster[c, t_row[b] + S-1-h, l_col[b] + j] - mean[c]) / std[c]     (fp32 subtraction, IEEE division)
 * `out` is channels-last (B, S, S, C), the image encoder's (B, C, S, S) input.  Window row h is raster row t_row + S-1-h,
 * the flip of t2h_blend_accumulate: row 0 is the southern edge, like row 0 of the cloud plane (pixel.py:105-111 adds the
 * two planes pixel by pixel).  Pixels outside the raster are written as NaN. */
int t2h_raster_windows(const float* raster, int C, int64_t rows, int64_t cols, const int32_t* t_row,
                       const int32_t* l_col, int n_tiles, int S, const float* mean, const float* std_dev, float* out,
                       t2h_stream_t stream);

/* ---- evaluation of a scene nDSM against the ground-truth DSM (evaluator.py:53-99: residual statistics per mask class,
 *      evaluator.py:83-95).  A pixel is valid when pred and gt are finite and (use_nodata) gt != nodata; r = pred - gt
 *      (one fp64 subtraction).  Class 0 is every valid pixel, class c + 1 the valid pixels with bit c of
 *      mask_bits[px] set (one byte per pixel, NULL when n_masks == 0, masks may overlap).  Per class:
 *        out_stats[class * 8 + 0..7] = mean, mae, rmse, min, max, median, medae, nmad;  out_count[class] = n
 *      median = numpy's rule (even n: (a + b) / 2 of the two middle values); medae = median |r|;
 *      nmad = 1.4826 * median |r - median(r)|.  count, min, max and the three medians are exact (MSD radix select on
 *      order-preserving 64-bit codes, 8-bit digits, 16 passes over the rasters); the sums use a reduction tree fixed by
 *      n, bitwise reproducible and independent of the other classes.  An empty class gives n = 0 and NaN elsewhere. */
size_t t2h_residual_stats_workspace_bytes(int64_t n_px, int n_masks);
int t2h_residual_stats(const double* pred, const double* gt, int64_t n_px, const uint8_t* mask_bits, int n_masks,
                       int use_nodata, double nodata, void* workspace, size_t workspace_bytes, double* out_stats,
                       int64_t* out_count, t2h_stream_t stream);

/* bias gradient: out[c] = sum_r g[r, c], two-stage and deterministic */
size_t t2h_colsum_workspace_bytes(int64_t rows, int n);
int t2h_colsum(const float* g, int64_t ld_g, int64_t rows, int n, void* workspace,
               size_t workspace_bytes, float* out, t2h_stream_t stream);

/* ---- one-call point-MLP blocks (SURVEY §8b: t2h_resblock_fwd/bwd, t2h_comm_mlp_fwd/bwd) ----------
 * COMPOSITIONS of the GEMM entry points above, enqueued on `stream` in the order the Python mirror issues them
 * (not single fused kernels, DESIGN.md §8.2): ReLU-on-load, the concat halves as two K sources, bias, the
 * shortcut / fc_c result as the residual of the last GEMM and the ReLU mask of the input gradients are fused into
 * the launches.  Weights are plain fp32 row-major [n_out][k_in]; the operand splits (3xTF32, or 3xFP16 for
 * n_out > 64 and K >= 128), the transposed weights of the input gradients and the row-split partials of the
 * weight gradients live in `workspace` (>= the matching *_workspace_bytes, which covers forward and backward).
 * Every dimension is a multiple of 4; with two sources k1 is a multiple of 32.
 *
 * ResnetBlockFC, block/resnet.py:46-54 (instances pointnet.py:37-39,73-79), x = [x1 | x2] (x2 nullable):
 *   net = fc_0(relu(x)),  out = shortcut(x) + fc_1(relu(net));  w_shortcut NULL = identity (k2 = 0, k1 = n_out).
 *   `net` (rows x n_h, the PRE-activation input of fc_1) is an output of the forward and an input of the backward.
 * backward: d_w1 = g^T relu(net), d_b1 = sum g;  g_net = (g w1) * (net > 0);  d_w0 = g_net^T relu(x), d_b0 = sum g_net;
 *   d_w_shortcut = g^T x;  d_x = (g_net w0) * (x > 0) + g w_shortcut (identity: + g).  d_x1 / d_x2 / d_b0 / d_b1 nullable. */
size_t t2h_resblock_workspace_bytes(int64_t rows, int k1, int k2, int n_h, int n_out, int has_shortcut);
int t2h_resblock_fwd(const float* x1, int64_t ld_x1, int k1, const float* x2, int64_t ld_x2, int k2,
                     int64_t rows, const float* w0, const float* b0, int n_h, const float* w1,
                     const float* b1, const float* w_shortcut, int n_out, void* workspace,
                     size_t workspace_bytes, float* net, int64_t ld_net, float* out, int64_t ld_out,
                     t2h_stream_t stream);
int t2h_resblock_bwd(const float* grad_out, int64_t ld_g, const float* x1, int64_t ld_x1, int k1,
                     const float* x2, int64_t ld_x2, int k2, const float* net, int64_t ld_net,
                     int64_t rows, const float* w0, int n_h, const float* w1, const float* w_shortcut,
                     int n_out, void* workspace, size_t workspace_bytes, float* d_x1, int64_t ld_dx1,
                     float* d_x2, int64_t ld_dx2, float* d_w0, float* d_b0, float* d_w1, float* d_b1,
                     float* d_w_shortcut, t2h_stream_t stream);

/* fc_comm + fc_c, encoder/alto.py:63-69,123-128 (and 164-170, 248-253):
 *   hidden = c w0^T + b0 (rows x 2C, pre-activation, an output),  out = relu(hidden) w2^T + b2 (+ c_last wc^T + bc);
 *   c_last NULL on the first level (C_prev ignored).
 * backward: d_w2 = g^T relu(hidden), d_b2 = sum g;  g_h = (g w2) * (hidden > 0);  d_w0 = g_h^T c, d_b0 = sum g_h;
 *   d_c = g_h w0;  d_wc = g^T c_last, d_bc = sum g, d_c_last = g wc.  d_c / d_c_last / bias gradients nullable. */
size_t t2h_comm_mlp_workspace_bytes(int64_t rows, int C, int C_prev);
int t2h_comm_mlp_fwd(const float* c, int64_t ld_c, int C, const float* c_last, int64_t ld_cl, int C_prev,
                     int64_t rows, const float* w0, const float* b0, const float* w2, const float* b2,
                     const float* wc, const float* bc, void* workspace, size_t workspace_bytes,
                     float* hidden, int64_t ld_hidden, float* out, int64_t ld_out, t2h_stream_t stream);
int t2h_comm_mlp_bwd(const float* grad_out, int64_t ld_g, const float* c, int64_t ld_c, int C,
                     const float* c_last, int64_t ld_cl, int C_prev, const float* hidden,
                     int64_t ld_hidden, int64_t rows, const float* w0, const float* w2, const float* wc,
                     void* workspace, size_t workspace_bytes, float* d_c, int64_t ld_dc, float* d_c_last,
                     int64_t ld_dcl, float* d_w0, float* d_b0, float* d_w2, float* d_b2, float* d_wc,
                     float* d_bc, t2h_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* T2H_H_ */
