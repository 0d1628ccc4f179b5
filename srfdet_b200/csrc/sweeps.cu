// Multi-sweep point input: mmdet3d 1.0.0rc6 LoadPointsFromMultiSweeps + PointsRangeFilter (restated, nothing
// vendored) as one fixed-capacity device stage.
//
// The sources (key frame first, then the chosen sweeps) are visited in order; inside a source, rows in index order.
// A row r < clamp(d_counts[s], 0, cap) of source s is kept unless
//   - SRF_SWEEP_REMOVE_CLOSE and |x| < r_close and |y| < r_close   (raw float32 coordinates, before the transform),
//   - a range is given and not lo < p < hi on x, y and z            (float32 values after the transform).
// SRF_SWEEP_TRANSFORM: xyz = fl32(fl32(R xyz) + t) with each product and sum rounded in float64 in the order
// ((x R_i0 + y R_i1) + z R_i2), no contraction -- numpy's float32 @ float64 then += float64 into a float32 array.
// SRF_SWEEP_TIME_LAG: column 4 reads d_lags[s].  Output column j is column cols[j] of the modified row.
//
// Two launches per call, a data-independent launch sequence, no host read and no allocation:
//   1. sweeps_count_kernel  one CTA per tile of SWEEP_TILE rows of one source: number of kept rows
//   2. sweeps_write_kernel  same tiles: offset = sum of the earlier tiles' counts, block-wide stable compaction;
//                           output rows of the tile's own range of the capacity that lie past the total get NaN
// The tile counts are few (Sigma cap / 1024), so every CTA of pass 2 re-reduces them instead of a third scan launch.
#include "common.cuh"

namespace srf {

constexpr int SWEEP_THREADS = 256;
constexpr int SWEEP_CHUNKS = 4;
constexpr int SWEEP_TILE = SWEEP_THREADS * SWEEP_CHUNKS;

struct SweepArgs {
  const float* pts[SRF_SWEEP_MAX_SOURCES];
  int32_t cap[SRF_SWEEP_MAX_SOURCES], ld[SRF_SWEEP_MAX_SOURCES], flags[SRF_SWEEP_MAX_SOURCES];
  int32_t tile0[SRF_SWEEP_MAX_SOURCES + 1];   // first tile of each source; tile0[n_src] = number of tiles
  int32_t row0[SRF_SWEEP_MAX_SOURCES];        // first capacity row of each source
  int32_t cols[SRF_SWEEP_MAX_COLS];
  int32_t n_src, n_cols, has_range;
  float lo[3], hi[3], radius;
};

__device__ __forceinline__ float rigid_row(float x, float y, float z, const double* __restrict__ m, double t) {
  const double r = __dadd_rn(__dadd_rn(__dmul_rn((double)x, m[0]), __dmul_rn((double)y, m[1])), __dmul_rn((double)z, m[2]));
  return __double2float_rn(__dadd_rn((double)__double2float_rn(r), t));
}

// keep test of row r of source s; with out != nullptr also the output row
__device__ __forceinline__ bool sweep_row(const SweepArgs& a, int s, int r, const double* __restrict__ poses,
                                          const float* __restrict__ lags, float* __restrict__ out) {
  const float* p = a.pts[s] + (size_t)r * a.ld[s];
  float x = __ldg(p), y = __ldg(p + 1), z = __ldg(p + 2);
  const int f = a.flags[s];
  if ((f & SRF_SWEEP_REMOVE_CLOSE) && fabsf(x) < a.radius && fabsf(y) < a.radius) return false;
  if (f & SRF_SWEEP_TRANSFORM) {
    const double* P = poses + (size_t)s * 12;
    const float tx = rigid_row(x, y, z, P + 0, __ldg(P + 9));
    const float ty = rigid_row(x, y, z, P + 3, __ldg(P + 10));
    const float tz = rigid_row(x, y, z, P + 6, __ldg(P + 11));
    x = tx;
    y = ty;
    z = tz;
  }
  if (a.has_range && !(a.lo[0] < x && x < a.hi[0] && a.lo[1] < y && y < a.hi[1] && a.lo[2] < z && z < a.hi[2]))
    return false;
  if (out) {
#pragma unroll
    for (int j = 0; j < SRF_SWEEP_MAX_COLS; ++j) {
      if (j >= a.n_cols) break;
      const int c = a.cols[j];
      out[j] = c == 0 ? x : c == 1 ? y : c == 2 ? z : (c == 4 && (f & SRF_SWEEP_TIME_LAG)) ? __ldg(lags + s) : __ldg(p + c);
    }
  }
  return true;
}

// tile -> (source, first local row, rows of the tile that hold valid points)
__device__ __forceinline__ void sweep_tile(const SweepArgs& a, const int32_t* __restrict__ counts, int tile, int& s,
                                           int& r0, int& n_valid, int& n_rows) {
  s = 0;
  while (s + 1 < a.n_src && a.tile0[s + 1] <= tile) ++s;
  r0 = (tile - a.tile0[s]) * SWEEP_TILE;
  const int n = min(max(__ldg(counts + s), 0), a.cap[s]);
  n_rows = min(SWEEP_TILE, a.cap[s] - r0);
  n_valid = max(0, min(SWEEP_TILE, n - r0));
}

__global__ void __launch_bounds__(SWEEP_THREADS) sweeps_count_kernel(SweepArgs a, const int32_t* __restrict__ counts,
                                                                     const double* __restrict__ poses,
                                                                     int32_t* __restrict__ tile_count) {
  int s, r0, n_valid, n_rows;
  sweep_tile(a, counts, blockIdx.x, s, r0, n_valid, n_rows);
  int kept = 0;
#pragma unroll
  for (int k = 0; k < SWEEP_CHUNKS; ++k) {
    const int i = k * SWEEP_THREADS + threadIdx.x;
    kept += (i < n_valid && sweep_row(a, s, r0 + i, poses, nullptr, nullptr)) ? 1 : 0;
  }
  __shared__ int s_sum[SWEEP_THREADS / 32];
#pragma unroll
  for (int o = 16; o; o >>= 1) kept += __shfl_xor_sync(0xffffffffu, kept, o);
  if ((threadIdx.x & 31) == 0) s_sum[threadIdx.x >> 5] = kept;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int w = 0; w < SWEEP_THREADS / 32; ++w) t += s_sum[w];
    tile_count[blockIdx.x] = t;
  }
}

__global__ void __launch_bounds__(SWEEP_THREADS) sweeps_write_kernel(SweepArgs a, const int32_t* __restrict__ counts,
                                                                     const double* __restrict__ poses,
                                                                     const float* __restrict__ lags,
                                                                     const int32_t* __restrict__ tile_count,
                                                                     float* __restrict__ out, int32_t* __restrict__ d_total) {
  __shared__ int s_a[SWEEP_THREADS / 32], s_b[SWEEP_THREADS / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n_tiles = a.tile0[a.n_src];
  int before = 0, all = 0;
  for (int t = threadIdx.x; t < n_tiles; t += SWEEP_THREADS) {
    const int c = __ldg(tile_count + t);
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
  for (int w = 0; w < SWEEP_THREADS / 32; ++w) {
    off += s_a[w];
    total += s_b[w];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) *d_total = total;

  int s, r0, n_valid, n_rows;
  sweep_tile(a, counts, blockIdx.x, s, r0, n_valid, n_rows);
  const int nc = a.n_cols;
  float row[SRF_SWEEP_MAX_COLS];
  for (int k = 0; k < SWEEP_CHUNKS; ++k) {
    const int i = k * SWEEP_THREADS + threadIdx.x;
    const bool keep = i < n_valid && sweep_row(a, s, r0 + i, poses, lags, row);
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    __syncthreads();                                   // s_a of the previous chunk has been read
    if (lane == 0) s_a[warp] = __popc(bal);
    __syncthreads();
    int pos = off + __popc(bal & ((1u << lane) - 1u)), chunk = 0;
    for (int w = 0; w < SWEEP_THREADS / 32; ++w) {
      pos += w < warp ? s_a[w] : 0;
      chunk += s_a[w];
    }
    if (keep) {
#pragma unroll
      for (int j = 0; j < SRF_SWEEP_MAX_COLS; ++j)
        if (j < nc) out[(size_t)pos * nc + j] = row[j];
    }
    off += chunk;
  }
  // NaN padding: the tile owns capacity rows [row0[s] + r0, + n_rows) of the output
  const int64_t g0 = (int64_t)a.row0[s] + r0;
  const float nan = __int_as_float(0x7fc00000);
  for (int e = threadIdx.x; e < n_rows * nc; e += SWEEP_THREADS) {
    const int64_t g = g0 + e / nc;
    if (g >= total) out[g * nc + e % nc] = nan;
  }
}

static int sweep_tiles(const srf_sweep_src* srcs, int n_src) {
  int64_t t = 0;
  for (int s = 0; s < n_src; ++s) t += cdiv(srcs[s].cap, SWEEP_TILE);
  return (int)t;
}

}  // namespace srf

using namespace srf;

extern "C" {

size_t srf_merge_sweeps_ws_bytes(const srf_sweep_src* srcs_host, int32_t n_src) {
  if (!srcs_host || n_src < 0 || n_src > SRF_SWEEP_MAX_SOURCES) return 0;
  return ((size_t)sweep_tiles(srcs_host, n_src) * 4 + 255) / 256 * 256 + 256;
}

int srf_merge_sweeps(const srf_sweep_src* srcs_host, int32_t n_src, const int32_t* d_counts, const double* d_poses,
                     const float* d_lags, const int32_t* cols_host, int32_t n_cols, const float range_host[6],
                     float close_radius, float* out, int32_t* d_total, void* ws, size_t ws_bytes, void* stream) {
  SRF_CHECK_ARG(d_total && cols_host, "srf_merge_sweeps: null arg");
  SRF_CHECK_ARG(n_src >= 0 && n_src <= SRF_SWEEP_MAX_SOURCES, "srf_merge_sweeps: need 0 <= n_src <= %d", SRF_SWEEP_MAX_SOURCES);
  SRF_CHECK_ARG(n_cols >= 3 && n_cols <= SRF_SWEEP_MAX_COLS, "srf_merge_sweeps: need 3 <= n_cols <= %d", SRF_SWEEP_MAX_COLS);
  SweepArgs a;
  a.n_src = n_src;
  a.n_cols = n_cols;
  a.has_range = range_host != nullptr;
  a.radius = close_radius;
  for (int j = 0; j < 3; ++j) {
    a.lo[j] = a.has_range ? range_host[j] : 0.f;
    a.hi[j] = a.has_range ? range_host[3 + j] : 0.f;
  }
  int max_col = 0;
  for (int j = 0; j < n_cols; ++j) {
    SRF_CHECK_ARG(cols_host[j] >= 0, "srf_merge_sweeps: negative column %d", cols_host[j]);
    a.cols[j] = cols_host[j];
    max_col = max(max_col, cols_host[j]);
  }
  int64_t tiles = 0, rows = 0;
  bool any_lag = false, any_pose = false;
  for (int s = 0; s < n_src; ++s) {
    const srf_sweep_src& src = srcs_host[s];
    SRF_CHECK_ARG(src.cap >= 0 && src.ld >= 3 && src.ld > max_col, "srf_merge_sweeps: source %d: need cap >= 0 and ld > every "
                  "column (ld %d, column %d)", s, src.ld, max_col);
    SRF_CHECK_ARG((src.flags & ~(SRF_SWEEP_TRANSFORM | SRF_SWEEP_TIME_LAG | SRF_SWEEP_REMOVE_CLOSE)) == 0,
                  "srf_merge_sweeps: source %d: unknown flags 0x%x", s, src.flags);
    SRF_CHECK_ARG(!(src.flags & SRF_SWEEP_TIME_LAG) || src.ld >= 5, "srf_merge_sweeps: source %d: time lag needs ld >= 5", s);
    SRF_CHECK_ARG(src.cap == 0 || src.points, "srf_merge_sweeps: source %d: null points", s);
    any_lag |= src.cap > 0 && (src.flags & SRF_SWEEP_TIME_LAG);
    any_pose |= src.cap > 0 && (src.flags & SRF_SWEEP_TRANSFORM);
    a.pts[s] = src.points;
    a.cap[s] = src.cap;
    a.ld[s] = src.ld;
    a.flags[s] = src.flags;
    a.tile0[s] = (int32_t)tiles;
    a.row0[s] = (int32_t)rows;
    tiles += cdiv(src.cap, SWEEP_TILE);
    rows += src.cap;
  }
  SRF_CHECK_ARG(rows < (int64_t)0x7fffffff, "srf_merge_sweeps: total capacity %lld too large", (long long)rows);
  a.tile0[n_src] = (int32_t)tiles;
  cudaStream_t st = (cudaStream_t)stream;
  if (tiles == 0) {
    SRF_CUDA(cudaMemsetAsync(d_total, 0, 4, st));
    return SRF_OK;
  }
  SRF_CHECK_ARG(d_counts && out && ws, "srf_merge_sweeps: null counts, output or workspace");
  SRF_CHECK_ARG(!any_pose || d_poses, "srf_merge_sweeps: null poses");
  SRF_CHECK_ARG(!any_lag || d_lags, "srf_merge_sweeps: null time lags");
  const size_t need = srf_merge_sweeps_ws_bytes(srcs_host, n_src);
  SRF_CHECK_ARG(ws_bytes >= need, "srf_merge_sweeps: workspace too small (%zu < %zu)", ws_bytes, need);
  int32_t* tile_count = (int32_t*)ws;
  SRF_COUNT(2);
  sweeps_count_kernel<<<(int)tiles, SWEEP_THREADS, 0, st>>>(a, d_counts, d_poses, tile_count);
  sweeps_write_kernel<<<(int)tiles, SWEEP_THREADS, 0, st>>>(a, d_counts, d_poses, d_lags, tile_count, out, d_total);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

}  // extern "C"
