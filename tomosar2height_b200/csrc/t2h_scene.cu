// Scene inference either side of the model forward (SURVEY §8f rank f2): tile crop + normalisation of the
// binned scene cloud, the normalised orthophoto windows of the tiles (models with the image branch), and
// flip * blend-window * accumulate of the predicted tiles into the scene rasters.
//
// Replace, per tile, the CPU boolean mask over a whole chunk (dataset.py:234 -> utils/crop_cloud.py:21-29),
// the 4x4 normalisation matmul + float cast + re-crop (dataset.py:243-278) and the python slice-add of
// generator.py:139-154.  The scene cloud is binned once by stride-sized cells (one sort); a tile then only
// looks at the <= 3 contiguous row ranges of the cells it overlaps.  Work items are 1024-candidate chunks of
// those ranges, listed on the host from the bin table: {tile, first candidate, count, chunk index in tile}.
//   pass 1 (t2h_tile_count): per chunk, the number of points that survive both crops; per tile, the minimum z
//          of the points that survive the first crop (z_shift: 'local_min', dataset.py:244-246)
//   pass 2 (t2h_tile_write): the survivors, normalised, in candidate order (stable: a chunk's slot is the
//          exclusive scan of the chunk counts, inside a chunk positions come from ballots)
// Everything is integer / comparison work plus one fp64 subtraction and division per coordinate -- HBM-bound.
#include "t2h_common.cuh"

namespace t2h {

constexpr int kCropThreads = 256;
constexpr int kCropChunk = 1024;  // candidates per work item

struct CropItem {
  int32_t tile;
  int32_t count;     // candidates in this item (<= kCropChunk)
  int64_t first;     // first candidate (row of the binned cloud)
};

// first crop: strictly inside the tile in world coordinates (crop_cloud.py:21-22, fp64 like the dataset);
// normalisation (dataset.py:252-276 without augmentation: (p - min) / patch, z relative to z_shift) in fp64,
// cast to fp32, second crop strictly inside the unit square (dataset.py:278)
__device__ __forceinline__ bool first_crop(double x, double y, double x0, double y0, double patch) {
  return x > x0 && x < x0 + patch && y > y0 && y < y0 + patch;
}
__device__ __forceinline__ bool second_crop(float nx, float ny) { return nx > 0.f && nx < 1.f && ny > 0.f && ny < 1.f; }

__global__ void __launch_bounds__(kCropThreads)
tile_count_kernel(const double* __restrict__ pts, const CropItem* __restrict__ items, const double* __restrict__ tile_xy,
                  double patch, int32_t* __restrict__ item_count, unsigned long long* __restrict__ tile_zmin) {
  __shared__ int s_cnt[kCropThreads / 32];
  __shared__ unsigned long long s_min[kCropThreads / 32];
  const CropItem it = items[blockIdx.x];
  const double x0 = tile_xy[2 * it.tile], y0 = tile_xy[2 * it.tile + 1];
  int cnt = 0;
  unsigned long long zmin = ~0ull;
  for (int i = threadIdx.x; i < it.count; i += kCropThreads) {
    const double* p = pts + (it.first + i) * 3;
    const double x = p[0], y = p[1];
    if (first_crop(x, y, x0, y0, patch)) {
      zmin = min(zmin, encode_f64(p[2]));
      cnt += second_crop((float)((x - x0) / patch), (float)((y - y0) / patch)) ? 1 : 0;
    }
  }
#pragma unroll
  for (int off = 16; off; off >>= 1) {
    cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
    zmin = min(zmin, __shfl_xor_sync(0xffffffffu, zmin, off));
  }
  if ((threadIdx.x & 31) == 0) { s_cnt[threadIdx.x >> 5] = cnt; s_min[threadIdx.x >> 5] = zmin; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kCropThreads / 32; ++w) { cnt += s_cnt[w]; zmin = min(zmin, s_min[w]); }
    item_count[blockIdx.x] = cnt;
    if (zmin != ~0ull) atomicMin(tile_zmin + it.tile, zmin);
  }
}

// out rows are (x, y, z, 0) fp32 -- the 16-byte rows the topology kernels read
__global__ void __launch_bounds__(kCropThreads)
tile_write_kernel(const double* __restrict__ pts, const CropItem* __restrict__ items, const double* __restrict__ tile_xy,
                  double patch, double z_scale, const int64_t* __restrict__ item_offset,
                  const unsigned long long* __restrict__ tile_zmin, float4* __restrict__ out) {
  __shared__ int s_warp[kCropThreads / 32];
  __shared__ int s_base;
  const CropItem it = items[blockIdx.x];
  const double x0 = tile_xy[2 * it.tile], y0 = tile_xy[2 * it.tile + 1];
  const double z_shift = decode_f64(tile_zmin[it.tile]);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_base = 0;
  __syncthreads();
  for (int i0 = 0; i0 < it.count; i0 += kCropThreads) {
    const int i = i0 + threadIdx.x;
    bool keep = false;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < it.count) {
      const double* p = pts + (it.first + i) * 3;
      const double x = p[0], y = p[1];
      if (first_crop(x, y, x0, y0, patch)) {
        v.x = (float)((x - x0) / patch);
        v.y = (float)((y - y0) / patch);
        v.z = (float)((p[2] - z_shift) / z_scale);
        keep = second_crop(v.x, v.y);
      }
    }
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) s_warp[warp] = __popc(m);
    __syncthreads();
    int before = s_base;
    for (int w = 0; w < warp; ++w) before += s_warp[w];
    if (keep) out[item_offset[blockIdx.x] + before + __popc(m & ((1u << lane) - 1u))] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
      int tot = 0;
      for (int w = 0; w < kCropThreads / 32; ++w) tot += s_warp[w];
      s_base += tot;
    }
    __syncthreads();
  }
}

// scene[r, c] += sum over the batch's tiles, IN TILE ORDER (the reference's sequential accumulation order), of
// (double) heights[b, S-1-i, j] * wx[j] * wy[i] with (i, j) = (r - t_row[b], c - l_col[b]); weight likewise.
// One thread per raster pixel of the batch's bounding box: overlapping tiles of one batch never race.
__global__ void __launch_bounds__(256)
blend_accumulate_kernel(const float* __restrict__ heights, int n_tiles, int S, const int32_t* __restrict__ t_row,
                        const int32_t* __restrict__ l_col, const double* __restrict__ wx, const double* __restrict__ wy,
                        int r0, int c0, int box_rows, int box_cols, int n_rows, int n_cols, double* __restrict__ dsm,
                        double* __restrict__ weight) {
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (int64_t)box_rows * box_cols) return;
  const int r = r0 + (int)(gid / box_cols), c = c0 + (int)(gid % box_cols);
  if (r < 0 || r >= n_rows || c < 0 || c >= n_cols) return;
  const int64_t px = (int64_t)r * n_cols + c;
  double acc = dsm[px], wacc = weight[px];  // running sums: the same additions, in the same order, as the reference
  bool hit = false;
  for (int b = 0; b < n_tiles; ++b) {
    const int i = r - t_row[b], j = c - l_col[b];
    if (i < 0 || i >= S || j < 0 || j >= S) continue;
    const double w = wx[j] * wy[i];
    // .flip(1) (generator.py:147); product and sum rounded separately, as `h_grid * patch_weight` then `+=` are
    acc = __dadd_rn(acc, __dmul_rn((double)heights[((int64_t)b * S + (S - 1 - i)) * S + j], w));
    wacc = __dadd_rn(wacc, w);
    hit = true;
  }
  if (hit) {
    dsm[px] = acc;
    weight[px] = wacc;
  }
}

// out[b, h, j, c] = (raster[c, t_row[b] + S-1-h, l_col[b] + j] - mean[c]) / std[c], channels-last (B, S, S, C).
// Row h of a window is raster row t_row + S-1-h: the same flip as blend_accumulate applies to the heights, so that
// window row 0 is the southern edge like row 0 of the cloud plane (y cell index).  A plain fp32 subtraction and an
// IEEE division, bitwise equal to the torch expression.  Pixels outside the raster are written as NaN (the caller
// checks coverage on the host; this only keeps a bad origin from reading out of bounds).
// One block row per output row (b, h), threads over j: every channel plane is read with coalesced loads, and the
// C interleaved stores of a warp cover one contiguous 128*C-byte run.
constexpr int kWindowThreads = 128;

__global__ void __launch_bounds__(kWindowThreads)
raster_windows_kernel(const float* __restrict__ raster, int C, int64_t rows, int64_t cols,
                      const int32_t* __restrict__ t_row, const int32_t* __restrict__ l_col, int S,
                      const float* __restrict__ mean, const float* __restrict__ std_dev, float* __restrict__ out) {
  const int bh = blockIdx.x;  // b * S + h
  const int b = bh / S, h = bh - b * S;
  const int j = blockIdx.y * kWindowThreads + threadIdx.x;
  if (j >= S) return;
  const int64_t r = (int64_t)t_row[b] + (S - 1 - h), c = (int64_t)l_col[b] + j;
  const bool inside = r >= 0 && r < rows && c >= 0 && c < cols;
  const int64_t plane = rows * cols;
  const float* src = raster + r * cols + c;
  float* dst = out + ((int64_t)bh * S + j) * C;
  for (int ch = 0; ch < C; ++ch)
    dst[ch] = inside ? __fdiv_rn(__fsub_rn(src[ch * plane], mean[ch]), std_dev[ch]) : __int_as_float(0x7fc00000);
}

}  // namespace t2h

using namespace t2h;

extern "C" int t2h_tile_count(const double* points, const void* items, int64_t n_items, const double* tile_xy,
                              double patch, int32_t* item_count, uint64_t* tile_zmin, t2h_stream_t stream) {
  if (n_items < 0 || patch <= 0.0 || (n_items > 0 && (!points || !items || !tile_xy || !item_count || !tile_zmin)))
    return T2H_ERR_INVALID_ARGUMENT;
  if (n_items == 0) return T2H_OK;
  tile_count_kernel<<<(unsigned)n_items, kCropThreads, 0, (cudaStream_t)stream>>>(
      points, (const CropItem*)items, tile_xy, patch, item_count, (unsigned long long*)tile_zmin);
  T2H_CHECK_LAUNCH();
  return T2H_OK;
}

extern "C" int t2h_tile_write(const double* points, const void* items, int64_t n_items, const double* tile_xy,
                              double patch, double z_scale, const int64_t* item_offset, const uint64_t* tile_zmin,
                              float* out_xyz0, t2h_stream_t stream) {
  if (n_items < 0 || patch <= 0.0 || z_scale <= 0.0 ||
      (n_items > 0 && (!points || !items || !tile_xy || !item_offset || !tile_zmin || !out_xyz0)))
    return T2H_ERR_INVALID_ARGUMENT;
  if (n_items == 0) return T2H_OK;
  tile_write_kernel<<<(unsigned)n_items, kCropThreads, 0, (cudaStream_t)stream>>>(
      points, (const CropItem*)items, tile_xy, patch, z_scale, item_offset, (const unsigned long long*)tile_zmin,
      (float4*)out_xyz0);
  T2H_CHECK_LAUNCH();
  return T2H_OK;
}

extern "C" int t2h_blend_accumulate(const float* heights, int n_tiles, int S, const int32_t* t_row, const int32_t* l_col,
                                    const double* wx, const double* wy, int r0, int c0, int box_rows, int box_cols,
                                    int n_rows, int n_cols, double* dsm, double* weight, t2h_stream_t stream) {
  if (n_tiles < 0 || S <= 0 || box_rows < 0 || box_cols < 0 || n_rows <= 0 || n_cols <= 0 ||
      (n_tiles > 0 && (!heights || !t_row || !l_col || !wx || !wy || !dsm || !weight)))
    return T2H_ERR_INVALID_ARGUMENT;
  const int64_t px = (int64_t)box_rows * box_cols;
  if (n_tiles == 0 || px == 0) return T2H_OK;
  blend_accumulate_kernel<<<(unsigned)((px + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      heights, n_tiles, S, t_row, l_col, wx, wy, r0, c0, box_rows, box_cols, n_rows, n_cols, dsm, weight);
  T2H_CHECK_LAUNCH();
  return T2H_OK;
}

extern "C" int t2h_raster_windows(const float* raster, int C, int64_t rows, int64_t cols, const int32_t* t_row,
                                  const int32_t* l_col, int n_tiles, int S, const float* mean, const float* std_dev,
                                  float* out, t2h_stream_t stream) {
  if (C <= 0 || rows <= 0 || cols <= 0 || n_tiles < 0 || S <= 0 ||
      (n_tiles > 0 && (!raster || !t_row || !l_col || !mean || !std_dev || !out)))
    return T2H_ERR_INVALID_ARGUMENT;
  if ((int64_t)n_tiles * S > 0x7fffffff) return T2H_ERR_UNSUPPORTED_SHAPE;
  if (n_tiles == 0) return T2H_OK;
  const dim3 grid((unsigned)(n_tiles * S), (unsigned)((S + kWindowThreads - 1) / kWindowThreads));
  raster_windows_kernel<<<grid, kWindowThreads, 0, (cudaStream_t)stream>>>(raster, C, rows, cols, t_row, l_col, S,
                                                                          mean, std_dev, out);
  T2H_CHECK_LAUNCH();
  return T2H_OK;
}
