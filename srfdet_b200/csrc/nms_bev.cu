// Multi-class BEV NMS of SRFDetHead.get_bboxes with use_nms=True (sparse_heads/srfdet_head.py:1269-1296:
// xywhr2xyxyr -> mmdet3d box3d_multiclass_nms -> mmcv nms_bev / nms_normal_bev), restated from the published
// sources of mmdet3d 1.0.0rc6 (core/post_processing/box3d_nms.py) and mmcv-full 1.7.0 (ops/iou3d.py, ops/nms.py,
// box_iou_rotated_utils.hpp); nothing is vendored.
//   srf_iou_bev     pairwise BEV IoU (rotated rectangles, or axis-aligned dx x dy when rotated = 0)
//   srf_nms_bev     per sample: IoU bitmask -> per-class greedy NMS -> class merge, max_num cut, range filter
//
// Footprint: the rectangle centred at (x, y) with extent dx along u = (cos yaw, sin yaw) and dy along
// v = (-sin yaw, cos yaw) -- LiDARInstance3DBoxes.bev as mmcv's rotated IoU sees it.  NOTE: this is the opposite
// rotation sense of boxes3d_to_corners3d / the RoI kernels (roi.cu), which rotate by -yaw; do not share code.
// IoU = area(A & B) / (area A + area B - area(A & B)), 0 when either area is below 1e-14; a box suppresses a
// lower-ranked one when IoU > thr (strict).  The rotated intersection is computed in fp32 on coordinates shifted
// to the pair's mid-centre (as mmcv does) by clipping one quad against the other (Sutherland-Hodgman, <= 8 vertices).
//
// srf_nms_bev is 3 launches with a data-independent launch sequence, no host synchronisation and no allocation:
//   1. nms_mask_kernel    one (k x k) "IoU > thr" bitmask per sample (the geometry does not depend on the class),
//                         64 x 64 pairs per CTA, each pair evaluated in one canonical order (lower index first)
//                         so the mask is symmetric bit for bit
//   2. nms_class_kernel   one CTA per (sample, class): candidates score > score_thr, bitonic sort by (score desc,
//                         index asc), the sample's mask staged in shared memory, greedy scan in blocks of 64
//                         candidates resolved in registers
//   3. nms_merge_kernel   one CTA per sample: class-major concatenation, the max_num cut (stable top-k: ties keep
//                         the class-major order), the post_center_range filter, fixed-capacity outputs + count
#include "common.cuh"

namespace srf {

constexpr int NMS_MAX_K = 1024;
constexpr int NMS_MAX_CLS = 32;
constexpr int NMS_MAX_WORDS = NMS_MAX_K / 64;
constexpr int NMS_CLASS_THREADS = 512;
constexpr int NMS_MERGE_THREADS = 1024;

struct BevBox {
  float x, y, dx, dy, c, s;
};

__device__ __forceinline__ BevBox load_bev(const float* __restrict__ row, bool rotated) {
  BevBox b;
  b.x = row[0];
  b.y = row[1];
  b.dx = row[3];
  b.dy = row[4];
  if (rotated) {
    sincosf(row[6], &b.s, &b.c);
  } else {
    b.c = 1.f;
    b.s = 0.f;
  }
  return b;
}

// area of the intersection of two convex quads given counter-clockwise (clip `a` by the 4 half-planes of `b`)
__device__ float quad_intersection_area(const float2 (&a)[4], const float2 (&b)[4]) {
  float2 poly[8], tmp[8];
  int n = 4;
#pragma unroll
  for (int i = 0; i < 4; ++i) poly[i] = a[i];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float2 p0 = b[e], p1 = b[(e + 1) & 3];
    const float ex = p1.x - p0.x, ey = p1.y - p0.y;
    int m = 0;
    for (int i = 0; i < n; ++i) {
      const float2 cur = poly[i], nxt = poly[i + 1 == n ? 0 : i + 1];
      const float dc = ex * (cur.y - p0.y) - ey * (cur.x - p0.x);
      const float dn = ex * (nxt.y - p0.y) - ey * (nxt.x - p0.x);
      if (dc >= 0.f && m < 8) tmp[m++] = cur;
      if ((dc >= 0.f) != (dn >= 0.f) && m < 8) {
        const float t = dc / (dc - dn);
        tmp[m++] = make_float2(cur.x + t * (nxt.x - cur.x), cur.y + t * (nxt.y - cur.y));
      }
    }
    if (m < 3) return 0.f;
    n = m;
    for (int i = 0; i < n; ++i) poly[i] = tmp[i];
  }
  float s = 0.f;
  for (int i = 0; i < n; ++i) {
    const float2 p = poly[i], q = poly[i + 1 == n ? 0 : i + 1];
    s += p.x * q.y - q.x * p.y;
  }
  return fmaxf(0.5f * s, 0.f);
}

__device__ __forceinline__ void bev_corners(const BevBox& b, float sx, float sy, float2 (&p)[4]) {
  const float cx = b.x - sx, cy = b.y - sy;
  const float hx = 0.5f * fabsf(b.dx), hy = 0.5f * fabsf(b.dy);
  const float ux = b.c * hx, uy = b.s * hx, vx = -b.s * hy, vy = b.c * hy;
  p[0] = make_float2(cx + ux + vx, cy + uy + vy);
  p[1] = make_float2(cx - ux + vx, cy - uy + vy);
  p[2] = make_float2(cx - ux - vx, cy - uy - vy);
  p[3] = make_float2(cx + ux - vx, cy + uy - vy);
}

// IoU of the BEV footprints (srf_iou_bev and the NMS mask call this one function)
__device__ float bev_iou(const BevBox& a, const BevBox& b, bool rotated) {
  const float area_a = a.dx * a.dy, area_b = b.dx * b.dy;
  if (area_a < 1e-14f || area_b < 1e-14f) return 0.f;
  // coordinates relative to the pair's mid-centre: small boxes far from the origin keep their fp32 precision
  const float sx = 0.5f * (a.x + b.x), sy = 0.5f * (a.y + b.y);
  float inter;
  if (!rotated) {
    const float ax = a.x - sx, ay = a.y - sy, bx = b.x - sx, by = b.y - sy;
    const float hax = 0.5f * fabsf(a.dx), hay = 0.5f * fabsf(a.dy), hbx = 0.5f * fabsf(b.dx), hby = 0.5f * fabsf(b.dy);
    const float w = fminf(ax + hax, bx + hbx) - fmaxf(ax - hax, bx - hbx);
    const float h = fminf(ay + hay, by + hby) - fmaxf(ay - hay, by - hby);
    inter = fmaxf(w, 0.f) * fmaxf(h, 0.f);
  } else {
    // circumscribed circles apart: no intersection (exact 0, no clipping)
    const float ddx = a.x - b.x, ddy = a.y - b.y;
    const float rr = 0.5f * (sqrtf(a.dx * a.dx + a.dy * a.dy) + sqrtf(b.dx * b.dx + b.dy * b.dy));
    if (ddx * ddx + ddy * ddy > rr * rr) return 0.f;
    float2 pa[4], pb[4];
    bev_corners(a, sx, sy, pa);
    bev_corners(b, sx, sy, pb);
    inter = quad_intersection_area(pa, pb);
  }
  return inter / (area_a + area_b - inter);
}

__global__ void iou_bev_kernel(const float* __restrict__ a, int m, int lda, const float* __restrict__ b, int n, int ldb, int rotated,
                               float* __restrict__ iou) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y * blockDim.y + threadIdx.y;
  if (i >= m || j >= n) return;
  iou[(size_t)i * n + j] = bev_iou(load_bev(a + (size_t)i * lda, rotated), load_bev(b + (size_t)j * ldb, rotated), rotated);
}

// mask[b][i][w] bit t: IoU(box i, box 64w + t) > thr (i != j); grid (words, words, bs), 64 threads = 64 rows
__global__ void __launch_bounds__(64) nms_mask_kernel(const float* __restrict__ boxes, int k, int dim, int rotated, float thr,
                                                      unsigned long long* __restrict__ mask) {
  __shared__ BevBox cols[64];
  const int b = blockIdx.z, W = gridDim.x;
  const int j0 = blockIdx.x * 64, i = blockIdx.y * 64 + threadIdx.x;
  const float* base = boxes + (size_t)b * k * dim;
  if (j0 + (int)threadIdx.x < k) cols[threadIdx.x] = load_bev(base + (size_t)(j0 + threadIdx.x) * dim, rotated);
  __syncthreads();
  if (i >= k) return;
  const BevBox r = load_bev(base + (size_t)i * dim, rotated);
  const int nj = min(64, k - j0);
  unsigned long long bits = 0;
  for (int t = 0; t < nj; ++t) {
    const int j = j0 + t;
    if (j == i) continue;
    const BevBox c = cols[t];
    // one call site, lower index first: (i, j) and (j, i) run the same instructions on the same operands
    if (bev_iou(i < j ? r : c, i < j ? c : r, rotated) > thr) bits |= 1ull << t;
  }
  mask[((size_t)b * k + i) * W + blockIdx.x] = bits;
}

// float -> uint32 with the same order (-0 == +0)
__device__ __forceinline__ unsigned ordered_bits(float s) {
  const unsigned u = __float_as_uint(s + 0.f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// one CTA per (class, sample): kept indices of the class in score order -> cls_idx[b][c][0 .. cls_cnt[b][c])
__global__ void __launch_bounds__(NMS_CLASS_THREADS) nms_class_kernel(const float* __restrict__ scores, int k, int n_cls, float score_thr,
                                                                      const unsigned long long* __restrict__ mask, int n2,
                                                                      int* __restrict__ cls_cnt, int* __restrict__ cls_idx) {
  extern __shared__ __align__(16) unsigned long long nms_smem[];
  const int c = blockIdx.x, b = blockIdx.y, W = (k + 63) / 64;
  unsigned long long* mask_s = nms_smem;                       // k x W
  unsigned long long* keys = mask_s + (size_t)k * W;           // n2: (~score, index), ascending = score descending
  unsigned long long* local = keys + n2;                       // n2: suppression row of a candidate within its block of 64
  __shared__ unsigned long long rem_s[NMS_MAX_WORDS];
  __shared__ int n_cand;
  const int tid = threadIdx.x, nt = blockDim.x;
  if (tid == 0) n_cand = 0;
  if (tid < NMS_MAX_WORDS) rem_s[tid] = 0;
  const unsigned long long* mg = mask + (size_t)b * k * W;
  for (int t = tid; t < k * W; t += nt) mask_s[t] = mg[t];
  __syncthreads();
  for (int i = tid; i < n2; i += nt) {
    unsigned long long key = ~0ull;
    if (i < k) {
      const float s = scores[((size_t)b * k + i) * n_cls + c];
      if (s > score_thr) {
        key = ((unsigned long long)~ordered_bits(s) << 32) | (unsigned)i;
        atomicAdd(&n_cand, 1);
      }
    }
    keys[i] = key;
  }
  __syncthreads();
  for (int size = 2; size <= n2; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = tid; t < n2 / 2; t += nt) {
        const int lo = 2 * t - (t & (stride - 1)), hi = lo + stride;
        const unsigned long long x = keys[lo], y = keys[hi];
        if ((x > y) == ((lo & size) == 0)) {
          keys[lo] = y;
          keys[hi] = x;
        }
      }
      __syncthreads();
    }
  }
  const int nc = n_cand;
  const int lane = tid & 31, warp = tid >> 5, n_warps = nt >> 5;
  // in-block suppression rows: bit q of local[r] = candidate r suppresses candidate (r & ~63) + q
  for (int r = warp; r < nc; r += n_warps) {
    const int r0 = r & ~63;
    const unsigned long long* row = mask_s + (size_t)(unsigned)keys[r] * W;
    bool s0 = false, s1 = false;
    if (r0 + lane < nc) {
      const unsigned j = (unsigned)keys[r0 + lane];
      s0 = (row[j >> 6] >> (j & 63)) & 1;
    }
    if (r0 + lane + 32 < nc) {
      const unsigned j = (unsigned)keys[r0 + lane + 32];
      s1 = (row[j >> 6] >> (j & 63)) & 1;
    }
    const unsigned lo = __ballot_sync(0xffffffffu, s0), hi = __ballot_sync(0xffffffffu, s1);
    if (lane == 0) local[r] = ((unsigned long long)hi << 32) | lo;
  }
  __syncthreads();
  if (warp != 0) return;
  // greedy scan: lane w < W owns word w of the removed set (also mirrored in rem_s for the block-entry test)
  unsigned long long rem = 0;
  int base = 0;
  int* out = cls_idx + ((size_t)b * n_cls + c) * k;
  for (int r0 = 0; r0 < nc; r0 += 64) {
    bool v0 = r0 + lane < nc, v1 = r0 + lane + 32 < nc;
    const unsigned j0 = v0 ? (unsigned)keys[r0 + lane] : 0u, j1 = v1 ? (unsigned)keys[r0 + lane + 32] : 0u;
    const bool a0 = v0 && !((rem_s[j0 >> 6] >> (j0 & 63)) & 1), a1 = v1 && !((rem_s[j1 >> 6] >> (j1 & 63)) & 1);
    unsigned long long alive = ((unsigned long long)__ballot_sync(0xffffffffu, a1) << 32) | __ballot_sync(0xffffffffu, a0);
    unsigned long long todo = alive;
    while (todo) {
      const int q = __ffsll((long long)todo) - 1;
      const unsigned long long later = q == 63 ? 0ull : (~0ull << (q + 1));
      alive &= ~(local[r0 + q] & later);
      if (lane < W) rem |= mask_s[(size_t)(unsigned)keys[r0 + q] * W + lane];
      todo = alive & later;
    }
    if ((alive >> lane) & 1) out[base + __popcll(alive & ((1ull << lane) - 1))] = (int)j0;
    if ((alive >> (lane + 32)) & 1) out[base + __popcll(alive & ((1ull << (lane + 32)) - 1))] = (int)j1;
    base += __popcll(alive);
    if (lane < W) rem_s[lane] = rem;
    __syncwarp();
  }
  if (lane == 0) cls_cnt[b * n_cls + c] = base;
}

// exclusive prefix of one flag per thread over the CTA; returns the CTA total through *total
__device__ __forceinline__ int block_exclusive_scan(bool flag, int* warp_sums, int* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
  const unsigned bal = __ballot_sync(0xffffffffu, flag);
  if (lane == 0) warp_sums[warp] = __popc(bal);
  __syncthreads();
  if (warp == 0) {
    const int v = lane < n_warps ? warp_sums[lane] : 0;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane < n_warps) warp_sums[lane] = incl - v;
    if (lane == 31) *total = incl;
  }
  __syncthreads();
  const int r = warp_sums[warp] + __popc(bal & ((1u << lane) - 1));
  __syncthreads();
  return r;
}

// one CTA per sample
__global__ void __launch_bounds__(NMS_MERGE_THREADS) nms_merge_kernel(const float* __restrict__ boxes, int k, int dim,
                                                                      const float* __restrict__ scores, int n_cls, int max_num,
                                                                      int has_range, float r0, float r1, float r2, float r3, float r4, float r5,
                                                                      const int* __restrict__ cls_cnt, const int* __restrict__ cls_idx,
                                                                      int* __restrict__ sel, float* __restrict__ out_boxes,
                                                                      float* __restrict__ out_scores, int* __restrict__ out_labels,
                                                                      int* __restrict__ out_index, int* __restrict__ d_count) {
  extern __shared__ __align__(16) float sc_s[];           // n_cls x k: scores of each class list, in list order
  __shared__ int cnt_s[NMS_MAX_CLS], off_s[NMS_MAX_CLS + 1], warp_sums[32], chunk_total;
  const int b = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
  if (tid == 0) {
    off_s[0] = 0;
    for (int c = 0; c < n_cls; ++c) {
      cnt_s[c] = cls_cnt[b * n_cls + c];
      off_s[c + 1] = off_s[c] + cnt_s[c];
    }
  }
  __syncthreads();
  const int total = off_s[n_cls];
  const int* idx_b = cls_idx + (size_t)b * n_cls * k;
  for (int t = tid; t < n_cls * k; t += nt) {
    const int c = t / k, j = t - c * k;
    if (j < cnt_s[c]) sc_s[t] = scores[((size_t)b * k + idx_b[t]) * n_cls + c];
  }
  __syncthreads();
  int* sel_b = sel + (size_t)b * n_cls * k;
  const bool cut = total > max_num;
  for (int t = tid; t < n_cls * k; t += nt) {
    const int c = t / k, j = t - c * k;
    if (j >= cnt_s[c]) continue;
    int slot = off_s[c] + j;
    if (cut) {
      if (j >= max_num) continue;
      // rank in (score desc, class-major position asc): earlier classes win ties, later classes lose them
      const float s = sc_s[t];
      int rank = j;
      for (int c2 = 0; c2 < n_cls; ++c2) {
        if (c2 == c) continue;
        const float* l = sc_s + (size_t)c2 * k;
        int lo = 0, hi = cnt_s[c2];            // first position whose score ranks after s
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (c2 < c ? l[mid] >= s : l[mid] > s) lo = mid + 1; else hi = mid;
        }
        rank += lo;
      }
      if (rank >= max_num) continue;
      slot = rank;
    }
    sel_b[slot] = t;
  }
  __syncthreads();
  const int n_sel = cut ? max_num : total;
  int count = 0;
  for (int s0 = 0; s0 < n_sel; s0 += nt) {
    const int s = s0 + tid;
    int t = 0, idx = 0;
    bool keep = false;
    if (s < n_sel) {
      t = sel_b[s];
      idx = idx_b[t];
      keep = true;
      if (has_range) {
        const float* bx = boxes + ((size_t)b * k + idx) * dim;
        keep = bx[0] >= r0 && bx[1] >= r1 && bx[2] >= r2 && bx[0] <= r3 && bx[1] <= r4 && bx[2] <= r5;
      }
    }
    const int pos = count + block_exclusive_scan(keep, warp_sums, &chunk_total);
    if (keep) {
      const size_t o = (size_t)b * max_num + pos;
      const float* bx = boxes + ((size_t)b * k + idx) * dim;
      for (int d = 0; d < dim; ++d) out_boxes[o * dim + d] = bx[d];
      out_scores[o] = sc_s[t];
      out_labels[o] = t / k;
      out_index[o] = idx;
    }
    count += chunk_total;
  }
  for (int r = count + tid; r < max_num; r += nt) {
    const size_t o = (size_t)b * max_num + r;
    for (int d = 0; d < dim; ++d) out_boxes[o * dim + d] = 0.f;
    out_scores[o] = 0.f;
    out_labels[o] = -1;
    out_index[o] = -1;
  }
  if (tid == 0) d_count[b] = count;
}

struct NmsWs {
  unsigned long long* mask;
  int *cls_cnt, *cls_idx, *sel;
  size_t bytes;
};

static inline size_t align256(size_t x) { return (x + 255) / 256 * 256; }

static NmsWs nms_ws(void* base, int bs, int k, int n_cls) {
  const size_t W = (size_t)(k + 63) / 64;
  const size_t m = align256((size_t)bs * k * W * 8), c = align256((size_t)bs * n_cls * 4), l = align256((size_t)bs * n_cls * k * 4);
  char* p = (char*)base;
  NmsWs w;
  w.mask = (unsigned long long*)p;
  w.cls_cnt = (int*)(p + m);
  w.cls_idx = (int*)(p + m + c);
  w.sel = (int*)(p + m + c + l);
  w.bytes = m + c + 2 * l;
  return w;
}

}  // namespace srf

using namespace srf;

extern "C" {

int srf_iou_bev(const float* a, int32_t m, int32_t lda, const float* b, int32_t n, int32_t ldb, int32_t rotated, float* iou, void* stream) {
  SRF_CHECK_ARG(a && b && iou && m >= 0 && n >= 0 && lda >= 7 && ldb >= 7, "srf_iou_bev: bad args (box rows need >= 7 columns)");
  if (m == 0 || n == 0) return SRF_OK;
  SRF_COUNT(1);
  iou_bev_kernel<<<dim3(cdiv(n, 16), cdiv(m, 16)), dim3(16, 16), 0, (cudaStream_t)stream>>>(a, m, lda, b, n, ldb, rotated, iou);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

size_t srf_nms_bev_ws_bytes(int32_t bs, int32_t k, int32_t n_cls) {
  if (bs < 1 || k < 1 || n_cls < 1) return 0;
  return nms_ws(nullptr, bs, k, n_cls).bytes;
}

int srf_nms_bev(const float* boxes, int32_t bs, int32_t k, int32_t dim, const float* scores, int32_t n_cls, float score_thr, float iou_thr,
                int32_t rotated, int32_t max_num, const float post_center_range[6], void* ws, size_t ws_bytes, float* out_boxes,
                float* out_scores, int32_t* out_labels, int32_t* out_index, int32_t* d_count, void* stream) {
  SRF_CHECK_ARG(boxes && scores && ws && out_boxes && out_scores && out_labels && out_index && d_count && bs >= 1 && k >= 1 && dim >= 7 &&
                    n_cls >= 1 && max_num >= 1,
                "srf_nms_bev: bad args");
  if (k > NMS_MAX_K || n_cls > NMS_MAX_CLS) {
    set_error("srf_nms_bev: at most %d boxes and %d classes per sample (got %d, %d)", NMS_MAX_K, NMS_MAX_CLS, k, n_cls);
    return SRF_ERR_UNSUPPORTED;
  }
  const NmsWs w = nms_ws(ws, bs, k, n_cls);
  SRF_CHECK_ARG(ws_bytes >= w.bytes, "srf_nms_bev: workspace of %zu B, need %zu (srf_nms_bev_ws_bytes)", ws_bytes, w.bytes);
  const int W = (k + 63) / 64;
  int n2 = 64;
  while (n2 < k) n2 <<= 1;
  const size_t smem_cls = ((size_t)k * W + 2 * (size_t)n2) * 8, smem_merge = (size_t)n_cls * k * 4;
  SRF_CUDA(cudaFuncSetAttribute(nms_class_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cls));
  SRF_CUDA(cudaFuncSetAttribute(nms_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_merge));
  cudaStream_t st = (cudaStream_t)stream;
  const float* r = post_center_range;
  SRF_COUNT(3);
  nms_mask_kernel<<<dim3(W, W, bs), 64, 0, st>>>(boxes, k, dim, rotated, iou_thr, w.mask);
  SRF_LAUNCH_CHECK();
  nms_class_kernel<<<dim3(n_cls, bs), NMS_CLASS_THREADS, smem_cls, st>>>(scores, k, n_cls, score_thr, w.mask, n2, w.cls_cnt, w.cls_idx);
  SRF_LAUNCH_CHECK();
  nms_merge_kernel<<<bs, NMS_MERGE_THREADS, smem_merge, st>>>(boxes, k, dim, scores, n_cls, max_num, r != nullptr, r ? r[0] : 0.f,
                                                               r ? r[1] : 0.f, r ? r[2] : 0.f, r ? r[3] : 0.f, r ? r[4] : 0.f,
                                                               r ? r[5] : 0.f, w.cls_cnt, w.cls_idx, w.sel, out_boxes, out_scores,
                                                               out_labels, out_index, d_count);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

}  // extern "C"
