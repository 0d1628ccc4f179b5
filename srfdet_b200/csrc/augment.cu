// Test-time augmentation of a point cloud (mmdet3d 1.0.0rc6 MultiScaleFlipAug3D around GlobalRotScaleTrans and
// RandomFlip3D, then an optional PointsRangeFilter; restated, nothing vendored): one fixed-capacity cloud in, A views
// of the same capacity out.
//
// Per view a, every row r < clamp(*d_count, 0, cap) of the input, in row order:
//   xyz *= scale[a]               (fp32, GlobalRotScaleTrans._scale_bbox_points with pcd_scale_factor)
//   flip bit 0 (horizontal):  y = -y,  flip bit 1 (vertical):  x = -x    (RandomFlip3D / LiDARPoints.flip)
//   kept unless a range is given and not lo < p < hi on x, y and z        (PointsRangeFilter, after both)
// Other columns are copied.  Kept rows are compacted stably into view a's block of cap rows; d_counts[a] = their number;
// rows past it are NaN, which every voxelizer drops as out of range.
//
// Two launches, grid (tiles, A): count, then write with the offset re-reduced from the tile counts (as sweeps.cu).
// No allocation and no host synchronisation: a captured call replays with a new count.
#include "common.cuh"

namespace srf {

constexpr int AUG_THREADS = 256;
constexpr int AUG_CHUNKS = 4;
constexpr int AUG_TILE = AUG_THREADS * AUG_CHUNKS;

struct AugArgs {
  float scale[SRF_AUG_MAX_VIEWS];
  int32_t flips[SRF_AUG_MAX_VIEWS];
  int32_t cap, n_cols, has_range;
  float lo[3], hi[3];
};

// keep test of row r in view a; with out != nullptr also the output row
__device__ __forceinline__ bool aug_row(const AugArgs& a, int v, const float* __restrict__ pts, int r, float* __restrict__ out) {
  const float* p = pts + (size_t)r * a.n_cols;
  const float s = a.scale[v];
  float x = __fmul_rn(__ldg(p), s), y = __fmul_rn(__ldg(p + 1), s), z = __fmul_rn(__ldg(p + 2), s);
  if (a.flips[v] & SRF_AUG_FLIP_HORIZONTAL) y = -y;
  if (a.flips[v] & SRF_AUG_FLIP_VERTICAL) x = -x;
  if (a.has_range && !(a.lo[0] < x && x < a.hi[0] && a.lo[1] < y && y < a.hi[1] && a.lo[2] < z && z < a.hi[2])) return false;
  if (out) {
    out[0] = x;
    out[1] = y;
    out[2] = z;
#pragma unroll
    for (int j = 3; j < SRF_AUG_MAX_COLS; ++j)
      if (j < a.n_cols) out[j] = __ldg(p + j);
  }
  return true;
}

__device__ __forceinline__ int aug_valid(const AugArgs& a, const int32_t* __restrict__ d_count) {
  return d_count ? min(max(__ldg(d_count), 0), a.cap) : a.cap;
}

__global__ void __launch_bounds__(AUG_THREADS) aug_count_kernel(AugArgs a, const float* __restrict__ pts,
                                                                const int32_t* __restrict__ d_count, int32_t* __restrict__ tile_count) {
  const int v = blockIdx.y, r0 = blockIdx.x * AUG_TILE;
  const int n_valid = max(0, min(AUG_TILE, aug_valid(a, d_count) - r0));
  int kept = 0;
#pragma unroll
  for (int k = 0; k < AUG_CHUNKS; ++k) {
    const int i = k * AUG_THREADS + threadIdx.x;
    kept += (i < n_valid && aug_row(a, v, pts, r0 + i, nullptr)) ? 1 : 0;
  }
  __shared__ int s_sum[AUG_THREADS / 32];
#pragma unroll
  for (int o = 16; o; o >>= 1) kept += __shfl_xor_sync(0xffffffffu, kept, o);
  if ((threadIdx.x & 31) == 0) s_sum[threadIdx.x >> 5] = kept;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int w = 0; w < AUG_THREADS / 32; ++w) t += s_sum[w];
    tile_count[(size_t)v * gridDim.x + blockIdx.x] = t;
  }
}

__global__ void __launch_bounds__(AUG_THREADS) aug_write_kernel(AugArgs a, const float* __restrict__ pts,
                                                                const int32_t* __restrict__ d_count,
                                                                const int32_t* __restrict__ tile_count, float* __restrict__ out,
                                                                int32_t* __restrict__ d_counts) {
  __shared__ int s_a[AUG_THREADS / 32], s_b[AUG_THREADS / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int v = blockIdx.y, n_tiles = gridDim.x;
  const int32_t* tc = tile_count + (size_t)v * n_tiles;
  int before = 0, all = 0;
  for (int t = threadIdx.x; t < n_tiles; t += AUG_THREADS) {
    const int c = __ldg(tc + t);
    all += c;
    before += t < (int)blockIdx.x ? c : 0;
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    before += __shfl_xor_sync(0xffffffffu, before, o);
    all += __shfl_xor_sync(0xffffffffu, all, o);
  }
  if (lane == 0) {
    s_a[warp] = before;
    s_b[warp] = all;
  }
  __syncthreads();
  int off = 0, total = 0;
  for (int w = 0; w < AUG_THREADS / 32; ++w) {
    off += s_a[w];
    total += s_b[w];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) d_counts[v] = total;

  const int r0 = blockIdx.x * AUG_TILE, nc = a.n_cols;
  const int n_valid = max(0, min(AUG_TILE, aug_valid(a, d_count) - r0));
  float* ov = out + (size_t)v * a.cap * nc;
  float row[SRF_AUG_MAX_COLS];
  for (int k = 0; k < AUG_CHUNKS; ++k) {
    const int i = k * AUG_THREADS + threadIdx.x;
    const bool keep = i < n_valid && aug_row(a, v, pts, r0 + i, row);
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    __syncthreads();                                   // s_a of the previous chunk has been read
    if (lane == 0) s_a[warp] = __popc(bal);
    __syncthreads();
    int pos = off + __popc(bal & ((1u << lane) - 1u)), chunk = 0;
    for (int w = 0; w < AUG_THREADS / 32; ++w) {
      pos += w < warp ? s_a[w] : 0;
      chunk += s_a[w];
    }
    if (keep) {
#pragma unroll
      for (int j = 0; j < SRF_AUG_MAX_COLS; ++j)
        if (j < nc) ov[(size_t)pos * nc + j] = row[j];
    }
    off += chunk;
  }
  // NaN padding: the tile owns rows [r0, r0 + AUG_TILE) of the view's capacity
  const int n_rows = min(AUG_TILE, a.cap - r0);
  const float nan = __int_as_float(0x7fc00000);
  for (int e = threadIdx.x; e < n_rows * nc; e += AUG_THREADS) {
    const int g = r0 + e / nc;
    if (g >= total) ov[(size_t)g * nc + e % nc] = nan;
  }
}

static inline size_t aug_ws_bytes(int32_t cap, int32_t n_views) {
  return ((size_t)cdiv(cap, AUG_TILE) * n_views * 4 + 255) / 256 * 256;
}

}  // namespace srf

using namespace srf;

extern "C" {

int srf_augment_points(const float* points, int32_t cap, int32_t n_cols, const int32_t* d_count, int32_t n_views,
                       const float* scales_host, const int32_t* flips_host, const float range_host[6], float* out,
                       int32_t* d_counts, void* ws, size_t* ws_bytes, void* stream) {
  SRF_CHECK_ARG(ws_bytes, "srf_augment_points: null ws_bytes");
  if (!ws) {
    SRF_CHECK_ARG(cap >= 0 && n_views >= 1 && n_views <= SRF_AUG_MAX_VIEWS, "srf_augment_points: bad capacity or views");
    *ws_bytes = aug_ws_bytes(cap, n_views);
    return SRF_OK;
  }
  SRF_CHECK_ARG(d_counts && scales_host && flips_host, "srf_augment_points: null arg");
  SRF_CHECK_ARG(n_views >= 1 && n_views <= SRF_AUG_MAX_VIEWS, "srf_augment_points: need 1 <= n_views <= %d", SRF_AUG_MAX_VIEWS);
  SRF_CHECK_ARG(n_cols >= 3 && n_cols <= SRF_AUG_MAX_COLS, "srf_augment_points: need 3 <= n_cols <= %d", SRF_AUG_MAX_COLS);
  SRF_CHECK_ARG(cap >= 0 && (int64_t)cap * n_cols * n_views < ((int64_t)1 << 40), "srf_augment_points: bad capacity %d", cap);
  AugArgs a;
  for (int v = 0; v < n_views; ++v) {
    SRF_CHECK_ARG((flips_host[v] & ~(SRF_AUG_FLIP_HORIZONTAL | SRF_AUG_FLIP_VERTICAL)) == 0,
                  "srf_augment_points: view %d: unknown flip flags 0x%x", v, flips_host[v]);
    a.scale[v] = scales_host[v];
    a.flips[v] = flips_host[v];
  }
  a.cap = cap;
  a.n_cols = n_cols;
  a.has_range = range_host != nullptr;
  for (int j = 0; j < 3; ++j) {
    a.lo[j] = a.has_range ? range_host[j] : 0.f;
    a.hi[j] = a.has_range ? range_host[3 + j] : 0.f;
  }
  cudaStream_t st = (cudaStream_t)stream;
  if (cap == 0) {
    SRF_CUDA(cudaMemsetAsync(d_counts, 0, (size_t)n_views * 4, st));
    return SRF_OK;
  }
  SRF_CHECK_ARG(points && out, "srf_augment_points: null points or output");
  const size_t need = aug_ws_bytes(cap, n_views);
  SRF_CHECK_ARG(*ws_bytes >= need, "srf_augment_points: workspace too small (%zu < %zu)", *ws_bytes, need);
  const dim3 grid(cdiv(cap, AUG_TILE), n_views);
  int32_t* tile_count = (int32_t*)ws;
  SRF_COUNT(2);
  aug_count_kernel<<<grid, AUG_THREADS, 0, st>>>(a, points, d_count, tile_count);
  aug_write_kernel<<<grid, AUG_THREADS, 0, st>>>(a, points, d_count, tile_count, out, d_counts);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

}  // extern "C"
