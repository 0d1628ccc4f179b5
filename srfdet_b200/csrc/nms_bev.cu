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
//
// srf_merge_aug_bev (mmdet3d merge_aug_bboxes_3d over the per-view results of test-time augmentation) is 4 launches
// with a data-independent launch sequence.  Up to SRF_MERGE_AUG_MAX_K = 4096 candidates per sample (views x rows), all
// possibly in one class: a k x k mask no longer fits shared memory, so it lives in the global workspace, in the order
// of the candidates sorted by (class, score desc, position asc), and only tiles that hold a same-class pair are built:
//   1. merge_aug_sort_kernel   one CTA per sample: the views' valid rows mapped back (bbox3d_mapping_back), sorted by
//                              (class, score desc, concatenated position asc) with a bitonic sort; class segments
//   2. merge_aug_mask_kernel   64 x 64 candidate tiles of the upper triangle: "same class and IoU > thr" bits
//   3. merge_aug_scan_kernel   one CTA per (class, sample): greedy scan of the class segment, blocks of 64 resolved in
//                              registers, the kept rows' mask words OR-ed into a shared removed set
//   4. merge_aug_final_kernel  one CTA per sample: the class-major kept lists sorted by (score desc, class-major
//                              position asc), the max_num cut, fixed-capacity outputs + count
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

// ------------------------------------------------------------------------------------------- test-time augmentation
constexpr int MERGE_AUG_THREADS = 1024;
constexpr int MERGE_AUG_SCAN_THREADS = 256;
constexpr int MERGE_AUG_MAX_WORDS = SRF_MERGE_AUG_MAX_K / 64;
constexpr float MERGE_AUG_PI = 3.14159265358979323846f;     // fl32(pi), as torch adds np.pi to a float32 tensor

struct MergeAugViews {
  float inv_scale[SRF_AUG_MAX_VIEWS];
  int32_t flips[SRF_AUG_MAX_VIEWS];
};

// bitonic sort of n2 (a power of two) keys in shared memory, ascending, by the whole CTA
__device__ __forceinline__ void block_bitonic_sort(unsigned long long* keys, int n2) {
  for (int size = 2; size <= n2; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = threadIdx.x; t < n2 / 2; t += blockDim.x) {
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
}

// key (class, score desc, position asc): class in bits 44.., ~score in bits 12..43, concatenated position in bits 0..11
__global__ void __launch_bounds__(MERGE_AUG_THREADS) merge_aug_sort_kernel(
    const float* __restrict__ boxes, const float* __restrict__ scores, const int* __restrict__ labels,
    const int* __restrict__ counts, int n_views, int m, int dim, MergeAugViews views, int n_cls, int n2,
    float* __restrict__ sbox, float* __restrict__ sscore, int* __restrict__ slab, int* __restrict__ cls_off) {
  extern __shared__ __align__(16) unsigned long long aug_keys[];
  __shared__ int voff[SRF_AUG_MAX_VIEWS + 1];
  const int b = blockIdx.x, tid = threadIdx.x, k = n_views * m;
  if (tid == 0) {
    voff[0] = 0;
    for (int a = 0; a < n_views; ++a) voff[a + 1] = voff[a] + min(max(counts[b * n_views + a], 0), m);
  }
  __syncthreads();
  const int n = voff[n_views];
  for (int p = tid; p < n2; p += blockDim.x) {
    unsigned long long key = ~0ull;
    if (p < n) {
      int a = 0;
      while (voff[a + 1] <= p) ++a;
      const size_t row = ((size_t)b * n_views + a) * m + (p - voff[a]);
      const int lab = labels[row];
      if (lab >= 0 && lab < n_cls) key = ((unsigned long long)lab << 44) | ((unsigned long long)(~ordered_bits(scores[row])) << 12) | (unsigned)p;
    }
    aug_keys[p] = key;
  }
  __syncthreads();
  block_bitonic_sort(aug_keys, n2);
  for (int i = tid; i < k; i += blockDim.x) {
    const unsigned long long key = aug_keys[i];
    const size_t o = (size_t)b * k + i;
    if (key == ~0ull) {
      slab[o] = n_cls;                      // past the valid candidates: a class of its own
      continue;
    }
    const int p = (int)(key & 0xfff);
    int a = 0;
    while (voff[a + 1] <= p) ++a;
    const size_t row = ((size_t)b * n_views + a) * m + (p - voff[a]);
    const bool hf = views.flips[a] & SRF_AUG_FLIP_HORIZONTAL, vf = views.flips[a] & SRF_AUG_FLIP_VERTICAL;
    const float inv_s = views.inv_scale[a];
    const float* src = boxes + row * dim;
    float* dst = sbox + o * dim;
    for (int d = 0; d < dim; ++d) {
      float x = src[d];
      if (d == 6) {                         // yaw: -yaw (horizontal), then -yaw + pi (vertical); not scaled
        if (hf) x = -x;
        if (vf) x = __fadd_rn(-x, MERGE_AUG_PI);
      } else {                              // y / vy (columns 1::7), x / vx (columns 0::7), then * fl32(1 / scale)
        if (hf && d % 7 == 1) x = -x;
        if (vf && d % 7 == 0) x = -x;
        x = __fmul_rn(x, inv_s);
      }
      dst[d] = x;
    }
    sscore[o] = scores[row];
    slab[o] = (int)(key >> 44);
  }
  // class c occupies sorted positions [cls_off[c], cls_off[c + 1]); cls_off[n_cls] = number of valid candidates
  for (int c = tid; c <= n_cls; c += blockDim.x) {
    int lo = 0, hi = n2;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if ((int)min(aug_keys[mid] >> 44, (unsigned long long)n_cls) < c) lo = mid + 1; else hi = mid;
    }
    cls_off[b * (NMS_MAX_CLS + 1) + c] = min(lo, k);
  }
}

// mask[b][i][w] bit t (sorted positions, j = 64w + t > i): same class and IoU(i, j) > thr.  Grid (W, W, bs); tiles below
// the diagonal and tiles whose row and column class ranges are disjoint are skipped: the scan reads only same-class
// bits, which lie in built tiles.
__global__ void __launch_bounds__(64) merge_aug_mask_kernel(const float* __restrict__ sbox, const int* __restrict__ slab, int k,
                                                            int dim, int n_cls, int rotated, float thr,
                                                            unsigned long long* __restrict__ mask) {
  __shared__ BevBox cols[64];
  __shared__ int col_lab[64];
  const int b = blockIdx.z, W = gridDim.x, R = blockIdx.y, C = blockIdx.x;
  if (C < R) return;
  const int* lab = slab + (size_t)b * k;
  const int i0 = R * 64, j0 = C * 64;
  const int lr0 = lab[i0], lr1 = lab[min(i0 + 63, k - 1)], lc0 = lab[j0], lc1 = lab[min(j0 + 63, k - 1)];
  if (lr0 >= n_cls || lc0 > lr1 || lr0 > lc1) return;
  const float* base = sbox + (size_t)b * k * dim;
  const int nj = min(64, k - j0);
  if ((int)threadIdx.x < nj) {
    col_lab[threadIdx.x] = lab[j0 + threadIdx.x];
    cols[threadIdx.x] = col_lab[threadIdx.x] < n_cls ? load_bev(base + (size_t)(j0 + threadIdx.x) * dim, rotated) : BevBox{};
  }
  __syncthreads();
  const int i = i0 + threadIdx.x;
  if (i >= k) return;
  const int li = lab[i];
  unsigned long long bits = 0;
  if (li < n_cls) {
    const BevBox r = load_bev(base + (size_t)i * dim, rotated);
    for (int t = 0; t < nj; ++t)
      if (j0 + t > i && col_lab[t] == li && bev_iou(r, cols[t], rotated) > thr) bits |= 1ull << t;
  }
  mask[((size_t)b * k + i) * W + C] = bits;
}

// one CTA per (class, sample): kept sorted positions of the class, in score order -> keep_idx[b][cls_off[c] + ...)
__global__ void __launch_bounds__(MERGE_AUG_SCAN_THREADS) merge_aug_scan_kernel(const int* __restrict__ cls_off, int k,
                                                                                const unsigned long long* __restrict__ mask,
                                                                                int* __restrict__ kept_cnt, int* __restrict__ keep_idx) {
  __shared__ unsigned long long rem_s[MERGE_AUG_MAX_WORDS], win_s[64], alive_s;
  const int c = blockIdx.x, b = blockIdx.y, n_cls = gridDim.x, tid = threadIdx.x;
  const int o = cls_off[b * (NMS_MAX_CLS + 1) + c], n = cls_off[b * (NMS_MAX_CLS + 1) + c + 1] - o;
  const int W = (k + 63) / 64;
  if (n <= 0) {
    if (tid == 0) kept_cnt[b * n_cls + c] = 0;
    return;
  }
  const int wlo = o >> 6, whi = (o + n - 1) >> 6;
  for (int w = wlo + tid; w <= whi; w += blockDim.x) rem_s[w] = 0;
  __syncthreads();
  const unsigned long long* mb = mask + (size_t)b * k * W;
  int* out = keep_idx + (size_t)b * k + o;
  int base = 0;
  for (int r0 = 0; r0 < n; r0 += 64) {
    const int g0 = o + r0, nb = min(64, n - r0), w0 = g0 >> 6, sh = g0 & 63;
    // window q: bit t = candidate r0 + q suppresses candidate r0 + t
    if (tid < nb) {
      const unsigned long long* row = mb + (size_t)(g0 + tid) * W;
      unsigned long long win = row[w0] >> sh;
      if (sh && w0 + 1 <= whi) win |= row[w0 + 1] << (64 - sh);
      win_s[tid] = nb == 64 ? win : win & ((1ull << nb) - 1);
    }
    __syncthreads();
    if (tid < 32) {
      const int lane = tid;
      const int q0 = lane, q1 = lane + 32;
      const bool a0 = q0 < nb && !((rem_s[(g0 + q0) >> 6] >> ((g0 + q0) & 63)) & 1);
      const bool a1 = q1 < nb && !((rem_s[(g0 + q1) >> 6] >> ((g0 + q1) & 63)) & 1);
      unsigned long long alive = ((unsigned long long)__ballot_sync(0xffffffffu, a1) << 32) | __ballot_sync(0xffffffffu, a0);
      unsigned long long todo = alive;
      while (todo) {
        const int q = __ffsll((long long)todo) - 1;
        const unsigned long long later = q == 63 ? 0ull : (~0ull << (q + 1));
        alive &= ~(win_s[q] & later);
        todo = alive & later;
      }
      if ((alive >> q0) & 1) out[base + __popcll(alive & ((1ull << q0) - 1))] = g0 + q0;
      if ((alive >> q1) & 1) out[base + __popcll(alive & ((1ull << q1) - 1))] = g0 + q1;
      if (lane == 0) alive_s = alive;
    }
    __syncthreads();
    const unsigned long long alive = alive_s;
    base += __popcll(alive);
    // the kept candidates' rows, words from the block's own to the segment's last, into the removed set
    const int nw = whi - w0 + 1;
    for (int e = tid; e < 64 * nw; e += blockDim.x) {
      const int q = e / nw, w = w0 + e % nw;
      if ((alive >> q) & 1) atomicOr(&rem_s[w], mb[(size_t)(g0 + q) * W + w]);
    }
    __syncthreads();
  }
  if (tid == 0) kept_cnt[b * n_cls + c] = base;
}

__global__ void __launch_bounds__(MERGE_AUG_THREADS) merge_aug_final_kernel(
    const float* __restrict__ sbox, const float* __restrict__ sscore, const int* __restrict__ slab, int k, int dim, int n_cls,
    int n2, const int* __restrict__ cls_off, const int* __restrict__ kept_cnt, const int* __restrict__ keep_idx, int max_num,
    float* __restrict__ out_boxes, float* __restrict__ out_scores, int* __restrict__ out_labels, int* __restrict__ d_count) {
  extern __shared__ __align__(16) unsigned long long aug_keys[];
  __shared__ int off_s[NMS_MAX_CLS + 1], cnt_s[NMS_MAX_CLS], total_s;
  const int b = blockIdx.x, tid = threadIdx.x;
  if (tid <= n_cls) off_s[tid] = cls_off[b * (NMS_MAX_CLS + 1) + tid];
  if (tid < n_cls) cnt_s[tid] = kept_cnt[b * n_cls + tid];
  __syncthreads();
  if (tid == 0) {
    int t = 0;
    for (int c = 0; c < n_cls; ++c) t += cnt_s[c];
    total_s = t;
  }
  const int* idx = keep_idx + (size_t)b * k;
  const float* sc = sscore + (size_t)b * k;
  // slot t of class c's segment holds a kept candidate when t - off[c] < kept[c]; key (score desc, slot asc)
  for (int t = tid; t < n2; t += blockDim.x) {
    unsigned long long key = ~0ull;
    if (t < off_s[n_cls]) {
      const int c = slab[(size_t)b * k + t];
      if (t - off_s[c] < cnt_s[c]) key = ((unsigned long long)(~ordered_bits(sc[idx[t]])) << 32) | (unsigned)t;
    }
    aug_keys[t] = key;
  }
  __syncthreads();
  block_bitonic_sort(aug_keys, n2);
  const int n_out = min(max_num, total_s);
  for (int r = tid; r < max_num; r += blockDim.x) {
    const size_t o = (size_t)b * max_num + r;
    if (r < n_out) {
      const int i = idx[(unsigned)aug_keys[r]];
      const float* bx = sbox + ((size_t)b * k + i) * dim;
      for (int d = 0; d < dim; ++d) out_boxes[o * dim + d] = bx[d];
      out_scores[o] = sc[i];
      out_labels[o] = slab[(size_t)b * k + i];
    } else {
      for (int d = 0; d < dim; ++d) out_boxes[o * dim + d] = 0.f;
      out_scores[o] = 0.f;
      out_labels[o] = -1;
    }
  }
  if (tid == 0) d_count[b] = n_out;
}

struct MergeAugWs {
  float *sbox, *sscore;
  int *slab, *cls_off, *kept_cnt, *keep_idx;
  unsigned long long* mask;
  size_t bytes;
};

static MergeAugWs merge_aug_ws(void* base, int bs, int k, int dim, int n_cls) {
  const size_t W = (size_t)(k + 63) / 64;
  const size_t sizes[7] = {align256((size_t)bs * k * dim * 4), align256((size_t)bs * k * 4), align256((size_t)bs * k * 4),
                           align256((size_t)bs * (NMS_MAX_CLS + 1) * 4), align256((size_t)bs * n_cls * 4),
                           align256((size_t)bs * k * 4), align256((size_t)bs * k * W * 8)};
  char* p = (char*)base;
  char* q[7];
  size_t total = 0;
  for (int i = 0; i < 7; ++i) {
    q[i] = p + total;
    total += sizes[i];
  }
  MergeAugWs w;
  w.sbox = (float*)q[0];
  w.sscore = (float*)q[1];
  w.slab = (int*)q[2];
  w.cls_off = (int*)q[3];
  w.kept_cnt = (int*)q[4];
  w.keep_idx = (int*)q[5];
  w.mask = (unsigned long long*)q[6];
  w.bytes = total;
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

int srf_merge_aug_bev(const float* boxes, const float* scores, const int32_t* labels, const int32_t* d_counts, int32_t bs,
                      int32_t n_views, int32_t m, int32_t dim, const float* inv_scales_host, const int32_t* flips_host,
                      int32_t n_cls, float iou_thr, int32_t rotated, int32_t max_num, void* ws, size_t* ws_bytes,
                      float* out_boxes, float* out_scores, int32_t* out_labels, int32_t* d_count, void* stream) {
  SRF_CHECK_ARG(ws_bytes && bs >= 1 && n_views >= 1 && m >= 1 && dim >= 7 && n_cls >= 1 && max_num >= 1, "srf_merge_aug_bev: bad args");
  const int64_t k = (int64_t)n_views * m;
  if (n_views > SRF_AUG_MAX_VIEWS || k > SRF_MERGE_AUG_MAX_K || n_cls > NMS_MAX_CLS) {
    set_error("srf_merge_aug_bev: at most %d views, %d candidates (views x rows) and %d classes per sample (got %d, %lld, %d)",
              SRF_AUG_MAX_VIEWS, SRF_MERGE_AUG_MAX_K, NMS_MAX_CLS, n_views, (long long)k, n_cls);
    return SRF_ERR_UNSUPPORTED;
  }
  const MergeAugWs w = merge_aug_ws(ws, bs, (int)k, dim, n_cls);
  if (!ws) {
    *ws_bytes = w.bytes;
    return SRF_OK;
  }
  SRF_CHECK_ARG(boxes && scores && labels && d_counts && inv_scales_host && flips_host && out_boxes && out_scores && out_labels && d_count,
                "srf_merge_aug_bev: null arg");
  SRF_CHECK_ARG(*ws_bytes >= w.bytes, "srf_merge_aug_bev: workspace of %zu B, need %zu", *ws_bytes, w.bytes);
  MergeAugViews v;
  for (int a = 0; a < n_views; ++a) {
    SRF_CHECK_ARG((flips_host[a] & ~(SRF_AUG_FLIP_HORIZONTAL | SRF_AUG_FLIP_VERTICAL)) == 0,
                  "srf_merge_aug_bev: view %d: unknown flip flags 0x%x", a, flips_host[a]);
    v.inv_scale[a] = inv_scales_host[a];
    v.flips[a] = flips_host[a];
  }
  int n2 = 64;
  while (n2 < k) n2 <<= 1;
  const int W = (int)((k + 63) / 64);
  cudaStream_t st = (cudaStream_t)stream;
  SRF_COUNT(4);
  merge_aug_sort_kernel<<<bs, MERGE_AUG_THREADS, (size_t)n2 * 8, st>>>(boxes, scores, labels, d_counts, n_views, m, dim, v, n_cls, n2,
                                                                       w.sbox, w.sscore, w.slab, w.cls_off);
  SRF_LAUNCH_CHECK();
  merge_aug_mask_kernel<<<dim3(W, W, bs), 64, 0, st>>>(w.sbox, w.slab, (int)k, dim, n_cls, rotated, iou_thr, w.mask);
  SRF_LAUNCH_CHECK();
  merge_aug_scan_kernel<<<dim3(n_cls, bs), MERGE_AUG_SCAN_THREADS, 0, st>>>(w.cls_off, (int)k, w.mask, w.kept_cnt, w.keep_idx);
  SRF_LAUNCH_CHECK();
  merge_aug_final_kernel<<<bs, MERGE_AUG_THREADS, (size_t)n2 * 8, st>>>(w.sbox, w.sscore, w.slab, (int)k, dim, n_cls, n2, w.cls_off,
                                                                        w.kept_cnt, w.keep_idx, max_num, out_boxes, out_scores,
                                                                        out_labels, d_count);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

}  // extern "C"
