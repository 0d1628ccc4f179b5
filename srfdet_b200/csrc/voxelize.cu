// Hard and dynamic voxelization (SURVEY.md 8 rows a1-a3).
//
// Reference semantics ([3P] mmcv 1.7.0 voxelization; call sites detectors/srfdet.py:221,238):
// points are visited in index order, a voxel is numbered by the index of its first point,
// keeps its first max_points points in index order, and voxels past max_voxels (in that
// numbering) are dropped.  mmcv's deterministic CUDA path gets there with an O(N*dup)
// scan and a <<<1,1>>> serial kernel; here the same result comes from order-independent
// parallel primitives:
//   1. hash insert of the voxel key with a 64-bit (key<<32 | min point index) entry
//      (atomicCAS to claim, atomicMin to keep the first point)           -> first-come owner
//   2. flag[i] = (i is the first point of its voxel); exclusive scan     -> voxel id = number
//      of first-points before i  == mmcv's running voxel_num
//   3. concurrent sorted insertion of each point index into its voxel's max_points slots
//      with an atomicMin cascade (final slot s = (s+1)-th smallest index, any schedule)
//   4. gather slots -> voxels / num_points / mean (HardSimpleVFE fused).
// Coordinates use __fsub_rn/__fdiv_rn + floorf so they are bit-identical to the CPU loop.
#include "common.cuh"

namespace srf {

struct GeomDev {
  float vs[3], lo[3];
  int32_t grid[3];
};

__device__ __forceinline__ bool point_cell(const float* __restrict__ p, const GeomDev& g, int& cx,
                                           int& cy, int& cz) {
  int c[3];
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    float q = __fdiv_rn(__fsub_rn(p[j], g.lo[j]), g.vs[j]);
    float f = floorf(q);
    // (int) of a NaN / huge float is undefined in C; treat as out of range
    if (!(f >= 0.f) || !(f < (float)g.grid[j])) return false;
    c[j] = (int)f;
  }
  cx = c[0];
  cy = c[1];
  cz = c[2];
  return true;
}

__global__ void dynamic_voxelize_kernel(const float* __restrict__ pts, int n, int c, GeomDev g,
                                        int batch_idx, int32_t* __restrict__ coors) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float* p = pts + (size_t)i * c;
    float xyz[3] = {__ldg(p), __ldg(p + 1), __ldg(p + 2)};
    int cx, cy, cz;
    bool ok = point_cell(xyz, g, cx, cy, cz);
    if (batch_idx >= 0) {
      int4 o = ok ? make_int4(batch_idx, cz, cy, cx) : make_int4(batch_idx, -1, -1, -1);
      reinterpret_cast<int4*>(coors)[i] = o;
    } else {
      int32_t* o = coors + (size_t)i * 3;
      o[0] = ok ? cz : -1;
      o[1] = ok ? cy : -1;
      o[2] = ok ? cx : -1;
    }
  }
}

// ---- hard voxelization ---------------------------------------------------------------
constexpr unsigned long long HASH_EMPTY = 0xffffffffffffffffull;

__device__ __forceinline__ uint32_t hash32(uint32_t k) {
  k ^= k >> 16;
  k *= 0x85ebca6bu;
  k ^= k >> 13;
  k *= 0xc2b2ae35u;
  k ^= k >> 16;
  return k;
}

// pass 1: key -> slot; entry = key<<32 | min(point index)
__global__ void hv_insert_kernel(const float* __restrict__ pts, int n, int c, GeomDev g,
                                 unsigned long long* __restrict__ table, uint32_t cap_mask,
                                 int32_t* __restrict__ point_slot, int32_t* __restrict__ point2voxel) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float* p = pts + (size_t)i * c;
    float xyz[3] = {__ldg(p), __ldg(p + 1), __ldg(p + 2)};
    int cx, cy, cz;
    int slot = -1;
    if (point_cell(xyz, g, cx, cy, cz)) {
      uint32_t key = (uint32_t)((cz * g.grid[1] + cy) * g.grid[0] + cx);
      unsigned long long mine = ((unsigned long long)key << 32) | (uint32_t)i;
      uint32_t h = hash32(key) & cap_mask;
      while (true) {
        unsigned long long cur = table[h];
        if (cur == HASH_EMPTY) {
          unsigned long long old = atomicCAS(table + h, HASH_EMPTY, mine);
          if (old == HASH_EMPTY) { slot = (int)h; break; }
          cur = old;
        }
        if ((uint32_t)(cur >> 32) == key) {
          atomicMin(table + h, mine);
          slot = (int)h;
          break;
        }
        h = (h + 1) & cap_mask;
      }
    }
    point_slot[i] = slot;
    if (point2voxel) point2voxel[i] = -1;
  }
}

// pass 2a: flag = point i opens its voxel
__global__ void hv_flag_kernel(const unsigned long long* __restrict__ table,
                               const int32_t* __restrict__ point_slot, int n,
                               uint32_t* __restrict__ flag) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    int s = point_slot[i];
    flag[i] = (s >= 0 && (uint32_t)(table[s] & 0xffffffffull) == (uint32_t)i) ? 1u : 0u;
  }
}

// pass 2c: first points publish their voxel id and coordinates
__global__ void hv_assign_kernel(const unsigned long long* __restrict__ table,
                                 const int32_t* __restrict__ point_slot, const uint32_t* __restrict__ flag,
                                 const uint32_t* __restrict__ rank, int n, GeomDev g, int max_voxels,
                                 int batch_idx, int32_t* __restrict__ slot2voxel,
                                 int32_t* __restrict__ coors, int32_t* __restrict__ d_voxel_num,
                                 const int32_t* __restrict__ d_total) {
  int gid = blockIdx.x * blockDim.x + threadIdx.x;
  if (gid == 0) *d_voxel_num = min(*d_total, max_voxels);
  for (int i = gid; i < n; i += gridDim.x * blockDim.x) {
    if (!flag[i]) continue;
    int s = point_slot[i];
    int v = (int)rank[i];
    if (v >= max_voxels) { slot2voxel[s] = -1; continue; }
    slot2voxel[s] = v;
    uint32_t key = (uint32_t)(table[s] >> 32);
    int cx = key % g.grid[0];
    key /= g.grid[0];
    int cy = key % g.grid[1];
    int cz = key / g.grid[1];
    if (batch_idx >= 0) {
      reinterpret_cast<int4*>(coors)[v] = make_int4(batch_idx, cz, cy, cx);
    } else {
      coors[(size_t)v * 3 + 0] = cz;
      coors[(size_t)v * 3 + 1] = cy;
      coors[(size_t)v * 3 + 2] = cx;
    }
  }
}

// pass 3: sorted insertion of the point index into its voxel's slot list (init 0x7f7f7f7f)
__global__ void hv_rank_kernel(const int32_t* __restrict__ point_slot, const int32_t* __restrict__ slot2voxel,
                               int n, int max_points, int32_t* __restrict__ lists) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    int s = point_slot[i];
    if (s < 0) continue;
    int v = slot2voxel[s];
    if (v < 0) continue;
    int32_t* L = lists + (size_t)v * max_points;
    int carry = i;
    for (int t = 0; t < max_points; ++t) {
      // cheap pre-check: a slot already holding a smaller index cannot take the carry
      int seen = *((volatile int32_t*)(L + t));
      if (seen < carry) continue;
      int old = atomicMin(L + t, carry);
      if (old == 0x7f7f7f7f) break;       // landed in a free slot
      if (old > carry) carry = old;        // displaced a larger index: keep bubbling it
    }
  }
}

// pass 4: one thread per voxel: num_points, mean, point2voxel; optional voxel payload
__global__ void hv_gather_kernel(const float* __restrict__ pts, int c, const int32_t* __restrict__ lists,
                                 int max_points, const int32_t* __restrict__ d_voxel_num,
                                 int32_t* __restrict__ num_points, float* __restrict__ mean,
                                 int32_t* __restrict__ point2voxel) {
  int m = *d_voxel_num;
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < m; v += gridDim.x * blockDim.x) {
    const int32_t* L = lists + (size_t)v * max_points;
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    int cnt = 0;
    for (int t = 0; t < max_points; ++t) {
      int i = L[t];
      if (i == 0x7f7f7f7f) break;
      ++cnt;
      if (point2voxel) point2voxel[i] = v;
      if (mean) {
        const float* p = pts + (size_t)i * c;
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (j < c) acc[j] += __ldg(p + j);
      }
    }
    num_points[v] = cnt;
    if (mean) {
      float fc = (float)cnt;
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (j < c) mean[(size_t)v * c + j] = __fdiv_rn(acc[j], fc);
    }
  }
}

// optional payload: one thread per (voxel, slot, channel) element, coalesced writes
__global__ void hv_payload_kernel(const float* __restrict__ pts, int c, const int32_t* __restrict__ lists,
                                  int max_points, const int32_t* __restrict__ d_voxel_num,
                                  float* __restrict__ voxels) {
  int64_t total = (int64_t)(*d_voxel_num) * max_points * c;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total;
       e += (int64_t)gridDim.x * blockDim.x) {
    int j = (int)(e % c);
    int64_t vs = e / c;
    int i = lists[vs];
    voxels[e] = (i == 0x7f7f7f7f) ? 0.f : __ldg(pts + (size_t)i * c + j);
  }
}

// ---- batched hard voxelization: compaction of per-sample blocks ---------------------------
// Block b of every array holds counts[b] valid rows at rows [b * block_rows, ...); they land at
// rows [sum_{j<b} counts[j], ...) of the packed output, in sample order.  Grid (x, n_blocks):
// one CTA row per block; each CTA recomputes its block's offset from the (few) device counts.
struct ConcatArrays {
  const uint32_t* src[SRF_CONCAT_MAX_ARRAYS];
  uint32_t* dst[SRF_CONCAT_MAX_ARRAYS];
  int32_t src_ld[SRF_CONCAT_MAX_ARRAYS], dst_ld[SRF_CONCAT_MAX_ARRAYS], width[SRF_CONCAT_MAX_ARRAYS];
  int32_t n;
};

__global__ void concat_counted_rows_kernel(const int32_t* __restrict__ counts, int n_blocks, int block_rows,
                                           ConcatArrays a, int32_t* __restrict__ d_total) {
  const int b = blockIdx.y;
  __shared__ int s_off, s_cnt;
  if (threadIdx.x == 0) {
    int off = 0;
    for (int j = 0; j < b; ++j) off += min(max(counts[j], 0), block_rows);
    const int cnt = min(max(counts[b], 0), block_rows);
    s_off = off;
    s_cnt = cnt;
    if (b == n_blocks - 1 && blockIdx.x == 0) *d_total = off + cnt;
  }
  __syncthreads();
  const int off = s_off, cnt = s_cnt;
  for (int k = 0; k < a.n; ++k) {
    const int w = a.width[k];
    const uint32_t* src = a.src[k] + (size_t)b * block_rows * a.src_ld[k];
    uint32_t* dst = a.dst[k] + (size_t)off * a.dst_ld[k];
    const int64_t total = (int64_t)cnt * w;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
      const int64_t r = e / w;
      const int j = (int)(e - r * w);
      dst[r * a.dst_ld[k] + j] = __ldg(src + r * a.src_ld[k] + j);
    }
  }
}

struct HvWs {
  unsigned long long* table;
  uint32_t cap;
  int32_t* point_slot;
  uint32_t* flag;
  uint32_t* rank;
  uint32_t* blocksum;
  int32_t* d_total;
  int32_t* slot2voxel;
  int32_t* lists;
  size_t bytes;
};

static uint32_t hv_capacity(int n) {
  uint32_t cap = 1024;
  while (cap < (uint32_t)n * 2u) cap <<= 1;
  return cap;
}

static HvWs hv_layout(void* base, int n, int max_points, int max_voxels) {
  HvWs w;
  w.cap = hv_capacity(n);
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off += (bytes + 255) / 256 * 256;
    return (char*)base + o;
  };
  w.table = (unsigned long long*)take((size_t)w.cap * 8);
  w.point_slot = (int32_t*)take((size_t)n * 4);
  w.flag = (uint32_t*)take((size_t)n * 4);
  w.rank = (uint32_t*)take((size_t)n * 4);
  w.blocksum = (uint32_t*)take((SCAN_BLOCKS + 4) * 4);
  w.d_total = (int32_t*)take(256);
  w.slot2voxel = (int32_t*)take((size_t)w.cap * 4);
  w.lists = (int32_t*)take((size_t)max_voxels * max_points * 4);
  w.bytes = off;
  return w;
}

}  // namespace srf

using namespace srf;

static int fill_geom(GeomDev* d, const srf_geom* g) {
  for (int j = 0; j < 3; ++j) {
    d->vs[j] = g->vs[j];
    d->lo[j] = g->lo[j];
    d->grid[j] = g->grid[j];
    if (!(g->vs[j] > 0.f) || g->grid[j] <= 0) return -1;
  }
  if ((int64_t)g->grid[0] * g->grid[1] * g->grid[2] >= (int64_t)0x7fffffff) return -1;
  return 0;
}

static int launch_grid(int64_t n, int threads) {
  int64_t g = (n + threads - 1) / threads;
  int64_t cap = (int64_t)sm_count() * 8;
  if (g > cap) g = cap;
  return g < 1 ? 1 : (int)g;
}

extern "C" {

int srf_geom_init(srf_geom* g, const float vs[3], const float range[6]) {
  SRF_CHECK_ARG(g && vs && range, "srf_geom_init: null arg");
  for (int j = 0; j < 3; ++j) {
    g->vs[j] = vs[j];
    g->lo[j] = range[j];
    g->hi[j] = range[3 + j];
    volatile float span = range[3 + j] - range[j];
    volatile float q = span / vs[j];
    g->grid[j] = (int32_t)lrintf(q);  // torch.round: half to even
    SRF_CHECK_ARG(g->grid[j] > 0, "srf_geom_init: empty grid on axis %d", j);
  }
  return SRF_OK;
}

int srf_dynamic_voxelize(const float* points, int32_t n, int32_t c, const srf_geom* g, int32_t batch_idx,
                         int32_t* coors, void* stream) {
  if (n == 0) return SRF_OK;
  SRF_CHECK_ARG(points && g && coors && n >= 0 && c >= 3, "srf_dynamic_voxelize: bad args");
  GeomDev gd;
  SRF_CHECK_ARG(fill_geom(&gd, g) == 0, "srf_dynamic_voxelize: bad geometry");
  if (n == 0) return SRF_OK;
  SRF_COUNT(1);
  dynamic_voxelize_kernel<<<launch_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(points, n, c, gd,
                                                                                 batch_idx, coors);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

size_t srf_hard_voxelize_ws_bytes(int32_t n, int32_t max_points, int32_t max_voxels) {
  if (n < 0 || max_points <= 0 || max_voxels <= 0) return 0;
  return hv_layout(nullptr, n, max_points, max_voxels).bytes;
}

int srf_hard_voxelize(const float* points, int32_t n, int32_t c, const srf_geom* g, int32_t max_points,
                      int32_t max_voxels, int32_t batch_idx, float* voxels, int32_t* coors,
                      int32_t* num_points, float* mean, int32_t* point2voxel, int32_t* d_voxel_num,
                      void* ws, size_t ws_bytes, void* stream) {
  SRF_CHECK_ARG(g && d_voxel_num, "srf_hard_voxelize: null arg");
  if (n == 0) {
    SRF_CUDA(cudaMemsetAsync(d_voxel_num, 0, 4, (cudaStream_t)stream));
    return SRF_OK;
  }
  SRF_CHECK_ARG(points && coors && num_points && ws, "srf_hard_voxelize: null arg");
  SRF_CHECK_ARG(n >= 0 && c >= 3 && c <= 8, "srf_hard_voxelize: need 3 <= c <= 8 (got %d)", c);
  SRF_CHECK_ARG(max_points > 0 && max_voxels > 0, "srf_hard_voxelize: max_points/max_voxels must be > 0");
  GeomDev gd;
  SRF_CHECK_ARG(fill_geom(&gd, g) == 0, "srf_hard_voxelize: bad geometry");
  HvWs w = hv_layout(ws, n, max_points, max_voxels);
  SRF_CHECK_ARG(ws_bytes >= w.bytes, "srf_hard_voxelize: workspace too small (%zu < %zu)", ws_bytes, w.bytes);
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) {
    SRF_CUDA(cudaMemsetAsync(d_voxel_num, 0, 4, st));
    return SRF_OK;
  }
  SRF_CUDA(cudaMemsetAsync(w.table, 0xff, (size_t)w.cap * 8, st));
  SRF_CUDA(cudaMemsetAsync(w.lists, 0x7f, (size_t)max_voxels * max_points * 4, st));
  int gp = launch_grid(n, 256);
  SRF_COUNT(voxels ? 6 : 5);
  hv_insert_kernel<<<gp, 256, 0, st>>>(points, n, c, gd, w.table, w.cap - 1, w.point_slot, point2voxel);
  hv_flag_kernel<<<gp, 256, 0, st>>>(w.table, w.point_slot, n, w.flag);
  int rc = scan_flags_launch(w.flag, w.rank, w.blocksum, n, w.d_total, 0, st);
  if (rc) return rc;
  hv_assign_kernel<<<gp, 256, 0, st>>>(w.table, w.point_slot, w.flag, w.rank, n, gd, max_voxels, batch_idx,
                                       w.slot2voxel, coors, d_voxel_num, w.d_total);
  hv_rank_kernel<<<gp, 256, 0, st>>>(w.point_slot, w.slot2voxel, n, max_points, w.lists);
  hv_gather_kernel<<<launch_grid(max_voxels, 128), 128, 0, st>>>(points, c, w.lists, max_points, d_voxel_num,
                                                                num_points, mean, point2voxel);
  if (voxels)
    hv_payload_kernel<<<launch_grid((int64_t)max_voxels * max_points * c, 256), 256, 0, st>>>(
        points, c, w.lists, max_points, d_voxel_num, voxels);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

int srf_concat_counted_rows(const int32_t* d_counts, int32_t n_blocks, int32_t block_rows, const srf_rows* arrays,
                            int32_t n_arrays, int32_t* d_total, void* stream) {
  SRF_CHECK_ARG(d_total && arrays, "srf_concat_counted_rows: null arg");
  SRF_CHECK_ARG(n_blocks >= 0 && n_blocks <= 65535 && block_rows > 0,
                "srf_concat_counted_rows: need 0 <= n_blocks <= 65535 and block_rows > 0");
  SRF_CHECK_ARG(n_arrays >= 1 && n_arrays <= SRF_CONCAT_MAX_ARRAYS, "srf_concat_counted_rows: need 1 <= n_arrays <= %d",
                SRF_CONCAT_MAX_ARRAYS);
  cudaStream_t st = (cudaStream_t)stream;
  if (n_blocks == 0) {
    SRF_CUDA(cudaMemsetAsync(d_total, 0, 4, st));
    return SRF_OK;
  }
  SRF_CHECK_ARG(d_counts, "srf_concat_counted_rows: null counts");
  ConcatArrays a;
  a.n = n_arrays;
  for (int k = 0; k < n_arrays; ++k) {
    const srf_rows& r = arrays[k];
    SRF_CHECK_ARG(r.src && r.dst && r.src != r.dst, "srf_concat_counted_rows: array %d: null or in-place", k);
    SRF_CHECK_ARG(r.width > 0 && r.width <= r.src_ld && r.width <= r.dst_ld,
                  "srf_concat_counted_rows: array %d: need 0 < width <= src_ld, dst_ld", k);
    a.src[k] = (const uint32_t*)r.src;
    a.dst[k] = (uint32_t*)r.dst;
    a.src_ld[k] = r.src_ld;
    a.dst_ld[k] = r.dst_ld;
    a.width[k] = r.width;
  }
  const int gx = max(1, launch_grid(block_rows, 256) / n_blocks);
  SRF_COUNT(1);
  concat_counted_rows_kernel<<<dim3(gx, n_blocks), 256, 0, st>>>(d_counts, n_blocks, block_rows, a, d_total);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

}  // extern "C"
