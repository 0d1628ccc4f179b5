// Region-feature extraction (SURVEY.md 8 rows a6-a8): box corners, the axis-aligned
// rectangle of the projected corners, mmdet's FPN level map and mmcv RoIAlign (7x7 bins,
// 2x2 samples, bilinear, avg, aligned=True), fused so that no RoI list, per-level
// nonzero()/index round trip or (n_cam,P,C,7,7) intermediate ever reaches HBM.
//
// Work split: one CTA per proposal (per (sample, proposal) for a batch); lanes own output bins (bin = lane, lane+32) and keep
// their 2x16 bilinear taps (offset, weight) in registers, warps stride over channels, so
// the taps are computed once per (proposal, camera) and each channel costs 32 coalesced-
// in-plane loads per lane.  The image variant accumulates the camera sum in registers.
#include "common.cuh"

namespace srf {

constexpr int POOL = 7;
constexpr int NBIN = POOL * POOL;

struct Pyr {
  const float* feat[4];
  int h[4], w[4];
  float scale[4];  // 1 / stride
  int n_levels, channels;
  int channels_last;  // maps are (n_img, H, W, C) in memory (torch channels_last) instead of (n_img, C, H, W)
};

struct OutSpec {
  void* ptr;
  int channel_last;  // (k,49,C') rows instead of (k,C,7,7)
  int enc;           // SRF_F32 or a 16-bit encoding (channel_last only); split rows are [hi | lo] halves of row_stride
  int lo_off;        // split encodings: elements from the hi half to the lo half (row_stride / 2)
  int row_stride;    // C' = channels of a destination row (>= C): lets two samplers fill one concatenated buffer
  int ch_offset;     // first destination channel
};

struct Taps {
  int off[16];
  float wt[16];
};

// mmdet SingleRoIExtractor.map_roi_levels: floor(log2(sqrt(w*h)/56 + 1e-6)) clamped to
// [0, n_levels-1]; evaluated with exact power-of-two thresholds instead of log2f.
__device__ __forceinline__ int roi_level(float x1, float y1, float x2, float y2, int n_levels) {
  float s = sqrtf((x2 - x1) * (y2 - y1));
  float t = s / 56.f + 1e-6f;
  int lvl = 0;
  float th = 2.f;
  for (int i = 1; i < n_levels; ++i, th *= 2.f) lvl += (t >= th) ? 1 : 0;
  return lvl;
}

// taps of one output bin: 4 samples x 4 corners, weights pre-divided by the sample count.
__device__ __forceinline__ void bin_taps(int bin, float x1s, float y1s, float bw, float bh, int H, int W, Taps& t) {
  const int ph = bin / POOL, pw = bin - ph * POOL;
#pragma unroll
  for (int iy = 0; iy < 2; ++iy) {
    float y = y1s + ph * bh + (iy + .5f) * bh / 2.f;
#pragma unroll
    for (int ix = 0; ix < 2; ++ix) {
      float x = x1s + pw * bw + (ix + .5f) * bw / 2.f;
      const int s = (iy * 2 + ix) * 4;
      if (y < -1.0f || y > (float)H || x < -1.0f || x > (float)W) {
#pragma unroll
        for (int q = 0; q < 4; ++q) { t.off[s + q] = 0; t.wt[s + q] = 0.f; }
        continue;
      }
      float yy = y <= 0.f ? 0.f : y, xx = x <= 0.f ? 0.f : x;
      int yl = (int)yy, xl = (int)xx, yh, xh;
      if (yl >= H - 1) { yh = yl = H - 1; yy = (float)yl; } else yh = yl + 1;
      if (xl >= W - 1) { xh = xl = W - 1; xx = (float)xl; } else xh = xl + 1;
      float ly = yy - yl, lx = xx - xl, hy = 1.f - ly, hx = 1.f - lx;
      t.off[s + 0] = yl * W + xl; t.wt[s + 0] = hy * hx;
      t.off[s + 1] = yl * W + xh; t.wt[s + 1] = hy * lx;
      t.off[s + 2] = yh * W + xl; t.wt[s + 2] = ly * hx;
      t.off[s + 3] = yh * W + xh; t.wt[s + 3] = ly * lx;
    }
  }
}

__device__ __forceinline__ float sample_bin(const float* __restrict__ plane, const Taps& t) {
  float acc = 0.f;
#pragma unroll
  for (int s = 0; s < 16; s += 4) {
    float v = t.wt[s] * __ldg(plane + t.off[s]) + t.wt[s + 1] * __ldg(plane + t.off[s + 1]) +
              t.wt[s + 2] * __ldg(plane + t.off[s + 2]) + t.wt[s + 3] * __ldg(plane + t.off[s + 3]);
    acc += v;
  }
  return acc * 0.25f;
}

__device__ __forceinline__ void store_bin(float* __restrict__ out, int k, int c, int bin, int C, int channel_last, float v) {
  if (channel_last) out[((size_t)k * NBIN + bin) * C + c] = v;
  else out[((size_t)k * C + c) * NBIN + bin] = v;
}

// one RoI (x1,y1,x2,y2 in input coordinates) of image `img` on its pyramid level.
__device__ __forceinline__ void roi_forward(const Pyr& p, int img, float x1, float y1, float x2, float y2,
                                            float* __restrict__ out, int k, int channel_last) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int lvl = roi_level(x1, y1, x2, y2, p.n_levels);
  const int H = p.h[lvl], W = p.w[lvl];
  const float sc = p.scale[lvl];
  const float x1s = x1 * sc - 0.5f, y1s = y1 * sc - 0.5f, x2s = x2 * sc - 0.5f, y2s = y2 * sc - 0.5f;
  const float bw = (x2s - x1s) / (float)POOL, bh = (y2s - y1s) / (float)POOL;
  Taps t0, t1;
  bin_taps(lane, x1s, y1s, bw, bh, H, W, t0);
  const bool has2 = lane + 32 < NBIN;
  bin_taps(has2 ? lane + 32 : 0, x1s, y1s, bw, bh, H, W, t1);
  const float* base = p.feat[lvl] + (size_t)img * p.channels * H * W;
  for (int c = warp; c < p.channels; c += nwarps) {
    const float* plane = base + (size_t)c * H * W;
    store_bin(out, k, c, lane, p.channels, channel_last, sample_bin(plane, t0));
    if (has2) store_bin(out, k, c, lane + 32, p.channels, channel_last, sample_bin(plane, t1));
  }
}

__global__ void __launch_bounds__(256) roi_extract_kernel(Pyr p, const float* __restrict__ rois, int k_total,
                                                         float* __restrict__ out, int channel_last) {
  const int k = blockIdx.x;
  if (k >= k_total) return;
  const float* r = rois + (size_t)k * 5;
  roi_forward(p, (int)r[0], r[1], r[2], r[3], r[4], out, k, channel_last);
}

// boxes3d_to_corners3d (core/bbox/util.py:84-176), bottom_center=False, ry=False.
// corner order: x = w/2*(+,-,-,+,+,-,-,+), y = l/2*(-,-,+,+,-,-,+,+), z = h/2*(-,-,-,-,+,+,+,+)
__device__ __forceinline__ void box_corners(float cx, float cy, float cz, float lw, float ll, float lh, float sn,
                                            float cs, float (*cor)[3]) {
  const float ry = atan2f(sn, cs);
  const float w = expf(lw), l = expf(ll), h = expf(lh);
  const float c = cosf(ry), s = sinf(ry);
  const float hw = w / 2.f, hl = l / 2.f, hh = h / 2.f;
  const float sx[8] = {1, -1, -1, 1, 1, -1, -1, 1};
  const float sy[8] = {-1, -1, 1, 1, -1, -1, 1, 1};
  const float sz[8] = {-1, -1, -1, -1, 1, 1, 1, 1};
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float xc = sx[i] * hw, yc = sy[i] * hl, zc = sz[i] * hh;
    cor[i][0] = cx + (xc * c + yc * s);
    cor[i][1] = cy + (-xc * s + yc * c);
    cor[i][2] = cz + zc;
  }
}

__global__ void corners_kernel(const float* __restrict__ boxes, int nb, int box_dim, float* __restrict__ corners) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nb) return;
  const float* b = boxes + (size_t)i * box_dim;
  float cor[8][3];
  box_corners(b[0], b[1], b[2], b[3], b[4], b[5], b[6], b[7], cor);
  float* o = corners + (size_t)i * 24;
#pragma unroll
  for (int j = 0; j < 8; ++j) { o[j * 3] = cor[j][0]; o[j * 3 + 1] = cor[j][1]; o[j * 3 + 2] = cor[j][2]; }
}

struct Range {
  float lo[3], span[3], vs[3];
};

__global__ void __launch_bounds__(256) bev_roi_kernel(Pyr p, float* __restrict__ boxes, int n_prop, int box_dim,
                                                     Range rg, int mutate, float* __restrict__ out, int channel_last,
                                                     float* __restrict__ rois_out) {
  const int k = blockIdx.x;  // b * n_prop + proposal
  float* b = boxes + (size_t)k * box_dim;
  // every thread reads the (still normalised) box before thread 0 overwrites the centre
  float bx[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) bx[j] = b[j];
  __syncthreads();
  const float cx = bx[0] * rg.span[0] + rg.lo[0], cy = bx[1] * rg.span[1] + rg.lo[1], cz = bx[2] * rg.span[2] + rg.lo[2];
  if (mutate && threadIdx.x == 0) { b[0] = cx; b[1] = cy; b[2] = cz; }
  float cor[8][3];
  box_corners(cx, cy, cz, bx[3], bx[4], bx[5], bx[6], bx[7], cor);
  float x1 = INFINITY, y1 = INFINITY, x2 = -INFINITY, y2 = -INFINITY;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float x = (cor[i][0] - rg.lo[0]) / rg.vs[0], y = (cor[i][1] - rg.lo[1]) / rg.vs[1];
    x1 = fminf(x1, x); x2 = fmaxf(x2, x); y1 = fminf(y1, y); y2 = fmaxf(y2, y);
  }
  const int img = k / n_prop;
  if (rois_out && threadIdx.x == 0) {
    float* r = rois_out + (size_t)k * 5;
    r[0] = (float)img; r[1] = x1; r[2] = y1; r[3] = x2; r[4] = y2;
  }
  roi_forward(p, img, x1, y1, x2, y2, out, k, channel_last);
}

// image branch: CPW = channels per warp held as register accumulators (camera sum).
// One CTA per (sample, proposal): k = b * n_prop + proposal.  Sample b sums its own cameras only: images
// b * n_cam + cam of the flattened pyramid, projected by lidar2img[b][cam] (B independent batch-1 calls, SURVEY.md 3.4).
template <int CPW>
__global__ void __launch_bounds__(256) img_roi_kernel(Pyr p, const float* __restrict__ boxes, int n_prop, int box_dim,
                                                     const float* __restrict__ lidar2img, int n_cam, Range rg,
                                                     float* __restrict__ out, int channel_last, float* __restrict__ rois_out) {
  const int k = blockIdx.x;
  const int smp = k / n_prop, prop = k - smp * n_prop, img0 = smp * n_cam;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const float* b = boxes + (size_t)k * box_dim;
  const float cx = b[0] * rg.span[0] + rg.lo[0], cy = b[1] * rg.span[1] + rg.lo[1], cz = b[2] * rg.span[2] + rg.lo[2];
  float cor[8][3];
  box_corners(cx, cy, cz, b[3], b[4], b[5], b[6], b[7], cor);
  float acc0[CPW], acc1[CPW];
#pragma unroll
  for (int i = 0; i < CPW; ++i) { acc0[i] = 0.f; acc1[i] = 0.f; }
  const bool has2 = lane + 32 < NBIN;
  for (int cam = 0; cam < n_cam; ++cam) {
    const int img = img0 + cam;
    const float* L = lidar2img + (size_t)img * 16;
    float x1 = INFINITY, y1 = INFINITY, x2 = -INFINITY, y2 = -INFINITY;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float X = cor[i][0], Y = cor[i][1], Z = cor[i][2];
      float u = __ldg(L + 0) * X + __ldg(L + 1) * Y + __ldg(L + 2) * Z + __ldg(L + 3);
      float v = __ldg(L + 4) * X + __ldg(L + 5) * Y + __ldg(L + 6) * Z + __ldg(L + 7);
      float d = __ldg(L + 8) * X + __ldg(L + 9) * Y + __ldg(L + 10) * Z + __ldg(L + 11);
      d = fmaxf(d, 1e-5f);
      u = u / d; v = v / d;
      x1 = fminf(x1, u); x2 = fmaxf(x2, u); y1 = fminf(y1, v); y2 = fmaxf(y2, v);
    }
    if (rois_out && threadIdx.x == 0) {
      float* r = rois_out + ((size_t)img * n_prop + prop) * 5;
      r[0] = (float)img; r[1] = x1; r[2] = y1; r[3] = x2; r[4] = y2;
    }
    const int lvl = roi_level(x1, y1, x2, y2, p.n_levels);
    const int H = p.h[lvl], W = p.w[lvl];
    const float sc = p.scale[lvl];
    const float x1s = x1 * sc - 0.5f, y1s = y1 * sc - 0.5f, x2s = x2 * sc - 0.5f, y2s = y2 * sc - 0.5f;
    // every sample lies inside [x1s,x2s]x[y1s,y2s]; RoIAlign reads 0 outside [-1,W]x[-1,H]
    if (x2s < -1.f || x1s > (float)W || y2s < -1.f || y1s > (float)H) continue;
    if (!(x2s >= x1s) || !(y2s >= y1s)) continue;  // NaN rectangle: mmdet assigns no level -> zeros
    const float bw = (x2s - x1s) / (float)POOL, bh = (y2s - y1s) / (float)POOL;
    Taps t0, t1;
    bin_taps(lane, x1s, y1s, bw, bh, H, W, t0);
    bin_taps(has2 ? lane + 32 : 0, x1s, y1s, bw, bh, H, W, t1);
    const float* base = p.feat[lvl] + (size_t)img * p.channels * H * W;
#pragma unroll
    for (int i = 0; i < CPW; ++i) {
      int c = warp + i * nwarps;
      if (c < p.channels) {
        const float* plane = base + (size_t)c * H * W;
        acc0[i] += sample_bin(plane, t0);
        if (has2) acc1[i] += sample_bin(plane, t1);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < CPW; ++i) {
    int c = warp + i * nwarps;
    if (c < p.channels) {
      store_bin(out, k, c, lane, p.channels, channel_last, acc0[i]);
      if (has2) store_bin(out, k, c, lane + 32, p.channels, channel_last, acc1[i]);
    }
  }
}

// ---------------------------------------------------------------- channels-last maps
// (n_img, H, W, C) memory order: a bilinear tap is one contiguous C-vector, so lanes own
// channels (float4 per lane = 128 channels per warp pass, one 512-byte coalesced request per
// tap), warps stride over the 49 bins and the (K,49,C) output is written with float4 stores.
struct RoiGeom {
  int lvl, H, W, live;
  float x1s, y1s, bw, bh;
};

__device__ __forceinline__ RoiGeom roi_geom(const Pyr& p, float x1, float y1, float x2, float y2) {
  RoiGeom g;
  g.lvl = roi_level(x1, y1, x2, y2, p.n_levels);
  g.H = p.h[g.lvl];
  g.W = p.w[g.lvl];
  const float sc = p.scale[g.lvl];
  g.x1s = x1 * sc - 0.5f;
  g.y1s = y1 * sc - 0.5f;
  const float x2s = x2 * sc - 0.5f, y2s = y2 * sc - 0.5f;
  g.bw = (x2s - g.x1s) / (float)POOL;
  g.bh = (y2s - g.y1s) / (float)POOL;
  g.live = !(x2s < -1.f || g.x1s > (float)g.W || y2s < -1.f || g.y1s > (float)g.H) && (x2s >= g.x1s) && (y2s >= g.y1s);
  return g;
}

// bilinear taps of ONE sample point (bin, iy, ix): 4 (offset, weight) pairs, weights already
// divided by the 4 samples of a bin.  Staged in shared memory once per (proposal, camera) so
// the channel loops only do  LDS + LDG.128 + 4 FFMA  per tap.  Offsets are BYTE offsets of the
// pixel's channel vector inside one image of the level (pixel * px_bytes, < 2^32: make_pyr), so
// a tap's address is one 32-bit-offset add (the 64-bit  pixel * C  product per tap was a third
// of the sampler's instructions).
__device__ __forceinline__ void sample_taps(int smp, const RoiGeom& g, uint32_t px_bytes, uint32_t* off, float* wt) {
  const int bin = smp >> 2, iy = (smp >> 1) & 1, ix = smp & 1;
  const int ph = bin / POOL, pw = bin - ph * POOL;
  const float y = g.y1s + ph * g.bh + (iy + .5f) * g.bh / 2.f;
  const float x = g.x1s + pw * g.bw + (ix + .5f) * g.bw / 2.f;
  const int H = g.H, W = g.W;
  if (y < -1.0f || y > (float)H || x < -1.0f || x > (float)W) {
#pragma unroll
    for (int q = 0; q < 4; ++q) { off[q] = 0; wt[q] = 0.f; }
    return;
  }
  float yy = y <= 0.f ? 0.f : y, xx = x <= 0.f ? 0.f : x;
  int yl = (int)yy, xl = (int)xx, yh, xh;
  if (yl >= H - 1) { yh = yl = H - 1; yy = (float)yl; } else yh = yl + 1;
  if (xl >= W - 1) { xh = xl = W - 1; xx = (float)xl; } else xh = xl + 1;
  const float ly = yy - yl, lx = xx - xl, hy = 1.f - ly, hx = 1.f - lx;
  off[0] = (uint32_t)(yl * W + xl) * px_bytes; wt[0] = hy * hx * 0.25f;
  off[1] = (uint32_t)(yl * W + xh) * px_bytes; wt[1] = hy * lx * 0.25f;
  off[2] = (uint32_t)(yh * W + xl) * px_bytes; wt[2] = ly * hx * 0.25f;
  off[3] = (uint32_t)(yh * W + xh) * px_bytes; wt[3] = ly * lx * 0.25f;
}

// resident CTAs per SM the compiler must leave room for / taps per batch of independent loads (A/B knobs)
#ifndef SRF_ROI_MINB
#define SRF_ROI_MINB 3
#endif
#ifndef SRF_ROI_TB
#define SRF_ROI_TB 16
#endif

constexpr int NTAP = NBIN * 16;   // taps per RoI: 49 bins x 4 samples x 4 corners

// accumulate one bin from staged taps into acc[NP] (float4 = 4 channels per lane per pass)
// The taps of a bin are loaded in batches of TB independent 16-byte loads per lane before any
// FMA consumes them (a load -> FMA -> load chain kept one request in flight per warp and left the
// kernel latency bound).  The inner loop is predicate-free: an out-of-range sample is staged as
// (offset 0, weight 0) -- its tap reads pixel 0 of the image and contributes 0 * v exactly --
// and lanes past the last channel read channel 0 (their accumulators are never stored).  A tap
// then costs  64-bit add + LDG.128 + 4 FFMA  (7 instructions; the earlier form with a 64-bit
// pixel * C product and per-tap zero-weight predicates ran at 20).  Accumulation order: tap 0..15.
template <int NP>
__device__ __forceinline__ void bin_accumulate_cl(const float* __restrict__ img_base, const uint32_t* __restrict__ s_off,
                                                  const float* __restrict__ s_wt, int bin, int C, int lane, float4* acc) {
  constexpr int TB = NP == 1 ? SRF_ROI_TB : 8;
  const char* lane_base[NP];
#pragma unroll
  for (int pss = 0; pss < NP; ++pss) {
    const int c = (pss * 32 + lane) * 4;
    lane_base[pss] = reinterpret_cast<const char*>(img_base) + (c < C ? c * 4 : 0);
  }
  // a bin whose 4 samples all fall outside the map (12 % of the bins of live cameras on the bench frame: boxes cut by the
  // image border) has 16 zero weights: nothing to add.  Weights are >= 0, so their sum tests them all; the branch is warp-uniform.
  float wall[16];
#pragma unroll
  for (int q = 0; q < 16; q += 4) *reinterpret_cast<float4*>(wall + q) = *reinterpret_cast<const float4*>(s_wt + bin * 16 + q);
  float wsum = 0.f;
#pragma unroll
  for (int q = 0; q < 16; ++q) wsum += wall[q];
  if (wsum == 0.f) return;
#pragma unroll
  for (int q0 = 0; q0 < 16; q0 += TB) {
    float w[TB];
    float4 v[TB][NP];
#pragma unroll
    for (int q = 0; q < TB; ++q) {
      w[q] = wall[q0 + q];
      const uint32_t off = s_off[bin * 16 + q0 + q];
#pragma unroll
      for (int pss = 0; pss < NP; ++pss) v[q][pss] = __ldg(reinterpret_cast<const float4*>(lane_base[pss] + off));
    }
#pragma unroll
    for (int q = 0; q < TB; ++q) {
#pragma unroll
      for (int pss = 0; pss < NP; ++pss) {
        acc[pss].x = fmaf(w[q], v[q][pss].x, acc[pss].x);
        acc[pss].y = fmaf(w[q], v[q][pss].y, acc[pss].y);
        acc[pss].z = fmaf(w[q], v[q][pss].z, acc[pss].z);
        acc[pss].w = fmaf(w[q], v[q][pss].w, acc[pss].w);
      }
    }
  }
}

template <int NP>
__device__ __forceinline__ void store_bin_cl(const OutSpec& o, int k, int bin, int C, int lane, const float4* acc) {
#pragma unroll
  for (int pss = 0; pss < NP; ++pss) {
    const int c = (pss * 32 + lane) * 4;
    if (c >= C) continue;
    if (o.channel_last) {
      const size_t e = ((size_t)k * NBIN + bin) * o.row_stride + o.ch_offset + c;
      if (o.enc != SRF_F32) {
        const bool f16 = enc_is_f16(o.enc);
        uint32_t h0, h1, l0, l1;
        split16x2(f16, acc[pss].x, acc[pss].y, h0, l0);
        split16x2(f16, acc[pss].z, acc[pss].w, h1, l1);
        *reinterpret_cast<uint2*>((uint16_t*)o.ptr + e) = make_uint2(h0, h1);
        if (enc_is_split(o.enc)) *reinterpret_cast<uint2*>((uint16_t*)o.ptr + e + o.lo_off) = make_uint2(l0, l1);
      } else {
        *reinterpret_cast<float4*>((float*)o.ptr + e) = acc[pss];
      }
    } else {
      float* op = (float*)o.ptr + ((size_t)k * C + c) * NBIN + bin;
      op[0] = acc[pss].x; op[NBIN] = acc[pss].y; op[2 * NBIN] = acc[pss].z; op[3 * NBIN] = acc[pss].w;
    }
  }
}

template <int NP>
__global__ void __launch_bounds__(256, NP == 1 ? SRF_ROI_MINB : 1) bev_roi_cl_kernel(Pyr p, float* __restrict__ boxes, const float* __restrict__ rois_in,
                                                        int n_prop, int box_dim, Range rg, int mutate, OutSpec out,
                                                        float* __restrict__ rois_out) {
  __shared__ __align__(16) uint32_t s_off[NTAP];
  __shared__ __align__(16) float s_wt[NTAP];
  const int k = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // box -> corners -> BEV rectangle -> level geometry on warp 0 only (atan2f / sinf / cosf / expf and eight rotated corners:
  // done by all 8 warps it was a fifth of the kernel's issued instructions); the other warps pick the result up from shared memory
  __shared__ RoiGeom s_g;
  __shared__ int s_img;
  if (warp == 0) {
    float x1, y1, x2, y2;
    int img;
    if (rois_in) {   // generic SingleRoIExtractor form
      const float* r = rois_in + (size_t)k * 5;
      img = (int)r[0]; x1 = r[1]; y1 = r[2]; x2 = r[3]; y2 = r[4];
    } else {
      float* b = boxes + (size_t)k * box_dim;
      float bx[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) bx[j] = b[j];
      __syncwarp();   // every lane has read the (still normalised) box before lane 0 overwrites the centre
      const float cx = bx[0] * rg.span[0] + rg.lo[0], cy = bx[1] * rg.span[1] + rg.lo[1], cz = bx[2] * rg.span[2] + rg.lo[2];
      if (mutate && lane == 0) { b[0] = cx; b[1] = cy; b[2] = cz; }
      float cor[8][3];
      box_corners(cx, cy, cz, bx[3], bx[4], bx[5], bx[6], bx[7], cor);
      x1 = INFINITY; y1 = INFINITY; x2 = -INFINITY; y2 = -INFINITY;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float x = (cor[i][0] - rg.lo[0]) / rg.vs[0], y = (cor[i][1] - rg.lo[1]) / rg.vs[1];
        x1 = fminf(x1, x); x2 = fmaxf(x2, x); y1 = fminf(y1, y); y2 = fmaxf(y2, y);
      }
      img = k / n_prop;
      if (rois_out && lane == 0) {
        float* r = rois_out + (size_t)k * 5;
        r[0] = (float)img; r[1] = x1; r[2] = y1; r[3] = x2; r[4] = y2;
      }
    }
    if (lane == 0) { s_g = roi_geom(p, x1, y1, x2, y2); s_img = img; }
  }
  __syncthreads();
  const RoiGeom g = s_g;
  const int img = s_img;
  if (threadIdx.x < NBIN * 4) sample_taps(threadIdx.x, g, (uint32_t)p.channels * 4u, s_off + threadIdx.x * 4, s_wt + threadIdx.x * 4);
  __syncthreads();
  const float* base = p.feat[g.lvl] + (size_t)img * g.H * g.W * p.channels;
  for (int bin = warp; bin < NBIN; bin += 8) {
    float4 acc[NP];
#pragma unroll
    for (int q = 0; q < NP; ++q) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    bin_accumulate_cl<NP>(base, s_off, s_wt, bin, p.channels, lane, acc);
    store_bin_cl<NP>(out, k, bin, p.channels, lane, acc);
  }
}

constexpr int IMG_MAX_CAM = 8;

template <int NP>
__global__ void __launch_bounds__(256, NP == 1 ? SRF_ROI_MINB : 1) img_roi_cl_kernel(Pyr p, const float* __restrict__ boxes, int n_prop, int box_dim,
                                                        const float* __restrict__ lidar2img, int n_cam, Range rg,
                                                        OutSpec out, float* __restrict__ rois_out) {
  extern __shared__ __align__(16) uint8_t sm_img[];
  uint32_t* s_off = reinterpret_cast<uint32_t*>(sm_img);       // [n_cam][NTAP]
  float* s_wt = reinterpret_cast<float*>(s_off + n_cam * NTAP);
  __shared__ RoiGeom sg[IMG_MAX_CAM];
  __shared__ const float* s_base[IMG_MAX_CAM];     // camera image of the RoI's level (resolved once: p.feat[] is indexed dynamically)
  const int k = blockIdx.x;   // b * n_prop + proposal (as img_roi_kernel)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // warp 0: lane = camera projects the box, resolves its level geometry, and the live cameras of this proposal are compacted
  // (1.2 of 6 on the bench frame): the tap staging and the bin loops only see those
  __shared__ int s_live[IMG_MAX_CAM];
  __shared__ int s_nlive;
  if (warp == 0) {
    bool live = false;
    if (lane < n_cam) {
      const int cam = lane;
      const int smp = k / n_prop, img = smp * n_cam + cam;
      const float* b = boxes + (size_t)k * box_dim;
      const float cx = b[0] * rg.span[0] + rg.lo[0], cy = b[1] * rg.span[1] + rg.lo[1], cz = b[2] * rg.span[2] + rg.lo[2];
      float cor[8][3];
      box_corners(cx, cy, cz, b[3], b[4], b[5], b[6], b[7], cor);
      const float* L = lidar2img + (size_t)img * 16;
      float x1 = INFINITY, y1 = INFINITY, x2 = -INFINITY, y2 = -INFINITY;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float X = cor[i][0], Y = cor[i][1], Z = cor[i][2];
        float u = __ldg(L + 0) * X + __ldg(L + 1) * Y + __ldg(L + 2) * Z + __ldg(L + 3);
        float v = __ldg(L + 4) * X + __ldg(L + 5) * Y + __ldg(L + 6) * Z + __ldg(L + 7);
        float d = __ldg(L + 8) * X + __ldg(L + 9) * Y + __ldg(L + 10) * Z + __ldg(L + 11);
        d = fmaxf(d, 1e-5f);
        u = u / d; v = v / d;
        x1 = fminf(x1, u); x2 = fmaxf(x2, u); y1 = fminf(y1, v); y2 = fmaxf(y2, v);
      }
      if (rois_out) {
        float* r = rois_out + ((size_t)img * n_prop + (k - smp * n_prop)) * 5;
        r[0] = (float)img; r[1] = x1; r[2] = y1; r[3] = x2; r[4] = y2;
      }
      const RoiGeom g = roi_geom(p, x1, y1, x2, y2);
      sg[cam] = g;
      s_base[cam] = p.feat[g.lvl] + (size_t)img * g.H * g.W * p.channels;   // per-image base in size_t; taps stay 32-bit inside it
      live = g.live != 0;
    }
    const unsigned m = __ballot_sync(0xffffffffu, live);
    if (live) s_live[__popc(m & ((1u << lane) - 1u))] = lane;
    if (lane == 0) s_nlive = __popc(m);
  }
  __syncthreads();
  const int n_live = s_nlive;
  for (int li = 0; li < n_live; ++li)
    if (threadIdx.x < NBIN * 4)
      sample_taps(threadIdx.x, sg[s_live[li]], (uint32_t)p.channels * 4u, s_off + li * NTAP + threadIdx.x * 4, s_wt + li * NTAP + threadIdx.x * 4);
  __syncthreads();
  for (int bin = warp; bin < NBIN; bin += 8) {
    float4 acc[NP];
#pragma unroll
    for (int q = 0; q < NP; ++q) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int li = 0; li < n_live; ++li)
      bin_accumulate_cl<NP>(s_base[s_live[li]], s_off + li * NTAP, s_wt + li * NTAP, bin, p.channels, lane, acc);
    store_bin_cl<NP>(out, k, bin, p.channels, lane, acc);
  }
}

static int make_pyr(Pyr* d, const srf_pyramid* p) {
  if (!p || p->n_levels < 1 || p->n_levels > 4 || p->channels < 1) return -1;
  for (int l = 0; l < 4; ++l) {
    bool live = l < p->n_levels;
    d->feat[l] = live ? p->feat[l] : nullptr;
    d->h[l] = live ? p->h[l] : 1;
    d->w[l] = live ? p->w[l] : 1;
    d->scale[l] = live ? 1.0f / p->stride[l] : 1.f;
    if (live && (!p->feat[l] || p->h[l] < 1 || p->w[l] < 1 || !(p->stride[l] > 0.f))) return -1;
  }
  d->n_levels = p->n_levels;
  d->channels = p->channels;
  d->channels_last = p->channels_last;
  if (p->channels_last && (p->channels % 4 != 0 || p->channels > 256)) return -1;
  if (p->channels_last)      // the samplers address a pixel by a 32-bit byte offset inside one image of a level
    for (int l = 0; l < p->n_levels; ++l)
      if ((unsigned long long)p->h[l] * p->w[l] * p->channels * 4ull >= (1ull << 32)) return -1;
  return 0;
}

static void make_range(Range* r, const float pc[6], const float vs[3]) {
  for (int j = 0; j < 3; ++j) {
    r->lo[j] = pc[j];
    r->span[j] = pc[3 + j] - pc[j];
    r->vs[j] = vs ? vs[j] : 1.f;
  }
}

}  // namespace srf

using namespace srf;

extern "C" {

int srf_boxes_to_corners(const float* boxes, int32_t nb, int32_t box_dim, float* corners, void* stream) {
  SRF_CHECK_ARG(boxes && corners && nb >= 0 && box_dim >= 8, "srf_boxes_to_corners: bad args");
  if (nb == 0) return SRF_OK;
  SRF_COUNT(1);
  corners_kernel<<<cdiv(nb, 128), 128, 0, (cudaStream_t)stream>>>(boxes, nb, box_dim, corners);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

static int make_out(OutSpec* o, const srf_roi_out* u, int channels, bool cl_maps, const char* who) {
  if (!u || !u->ptr) { set_error("%s: null output", who); return SRF_ERR_ARG; }
  o->ptr = u->ptr;
  o->channel_last = u->channel_last;
  o->enc = u->dtype;
  const int parts = enc_is_split(o->enc) ? 2 : 1;
  o->row_stride = u->row_stride > 0 ? u->row_stride : parts * channels;
  o->lo_off = o->row_stride / 2;
  o->ch_offset = u->ch_offset;
  if (o->enc != SRF_F32 && !enc_is_16(o->enc)) { set_error("%s: bad output dtype", who); return SRF_ERR_ARG; }
  const bool plain = o->enc == SRF_F32 && o->row_stride == channels && o->ch_offset == 0;
  if (!plain && !(cl_maps && o->channel_last)) {
    set_error("%s: 16-bit / strided output needs channel_last output and channels_last feature maps", who);
    return SRF_ERR_UNSUPPORTED;
  }
  if (o->row_stride / parts < o->ch_offset + channels || (o->row_stride % (4 * parts)) || (o->ch_offset % 4)) {
    set_error("%s: bad output row stride / channel offset", who);
    return SRF_ERR_ARG;
  }
  return SRF_OK;
}

int srf_roi_extract(const srf_pyramid* p, const float* rois, int32_t k, float* out, int32_t channel_last, void* stream) {
  Pyr d;
  SRF_CHECK_ARG(make_pyr(&d, p) == 0, "srf_roi_extract: bad pyramid");
  SRF_CHECK_ARG(rois && out && k >= 0, "srf_roi_extract: bad args");
  if (k == 0) return SRF_OK;
  SRF_COUNT(1);
  if (d.channels_last) {
    Range rg = {};
    OutSpec o{out, channel_last, SRF_F32, 0, d.channels, 0};
    if (d.channels <= 128) bev_roi_cl_kernel<1><<<k, 256, 0, (cudaStream_t)stream>>>(d, nullptr, rois, 1, 0, rg, 0, o, nullptr);
    else bev_roi_cl_kernel<2><<<k, 256, 0, (cudaStream_t)stream>>>(d, nullptr, rois, 1, 0, rg, 0, o, nullptr);
    SRF_LAUNCH_CHECK();
    return SRF_OK;
  }
  roi_extract_kernel<<<k, 256, 0, (cudaStream_t)stream>>>(d, rois, k, out, channel_last);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

int srf_bev_roi_features(const srf_pyramid* p, float* boxes, int32_t batch, int32_t n_prop, int32_t box_dim,
                         const float pc_range[6], const float voxel_size[3], int32_t mutate, const srf_roi_out* out_spec,
                         float* rois_out, void* stream) {
  Pyr d;
  SRF_CHECK_ARG(make_pyr(&d, p) == 0, "srf_bev_roi_features: bad pyramid");
  SRF_CHECK_ARG(boxes && pc_range && voxel_size && batch >= 1 && n_prop >= 0 && box_dim >= 8, "srf_bev_roi_features: bad args");
  OutSpec o;
  { int rc = make_out(&o, out_spec, d.channels, d.channels_last != 0, "srf_bev_roi_features"); if (rc) return rc; }
  float* out = (float*)o.ptr;
  const int channel_last = o.channel_last;
  if (n_prop == 0) return SRF_OK;
  Range rg;
  make_range(&rg, pc_range, voxel_size);
  SRF_COUNT(1);
  if (d.channels_last) {
    if (d.channels <= 128) bev_roi_cl_kernel<1><<<batch * n_prop, 256, 0, (cudaStream_t)stream>>>(d, boxes, nullptr, n_prop, box_dim, rg, mutate, o, rois_out);
    else bev_roi_cl_kernel<2><<<batch * n_prop, 256, 0, (cudaStream_t)stream>>>(d, boxes, nullptr, n_prop, box_dim, rg, mutate, o, rois_out);
    SRF_LAUNCH_CHECK();
    return SRF_OK;
  }
  bev_roi_kernel<<<batch * n_prop, 256, 0, (cudaStream_t)stream>>>(d, boxes, n_prop, box_dim, rg, mutate, out, channel_last, rois_out);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

int srf_img_roi_features(const srf_pyramid* p, const float* boxes, int32_t batch, int32_t n_prop, int32_t box_dim,
                         const float* lidar2img, int32_t n_cam, const float pc_range[6], const srf_roi_out* out_spec,
                         float* rois_out, void* stream) {
  Pyr d;
  SRF_CHECK_ARG(make_pyr(&d, p) == 0, "srf_img_roi_features: bad pyramid");
  SRF_CHECK_ARG(batch >= 1, "srf_img_roi_features: batch must be >= 1 (got %d)", batch);
  SRF_CHECK_ARG(boxes && lidar2img && pc_range && n_prop >= 0 && box_dim >= 8 && n_cam >= 1, "srf_img_roi_features: bad args");
  SRF_CHECK_ARG((long long)batch * n_prop <= 0x7fffffffLL && (long long)batch * n_cam <= 0x7fffffffLL,
                "srf_img_roi_features: batch %d x %d proposals / %d cameras overflows", batch, n_prop, n_cam);
  OutSpec o;
  { int rc = make_out(&o, out_spec, d.channels, d.channels_last != 0, "srf_img_roi_features"); if (rc) return rc; }
  float* out = (float*)o.ptr;
  const int channel_last = o.channel_last;
  SRF_CHECK_ARG(d.channels <= 256, "srf_img_roi_features: at most 256 channels (got %d)", d.channels);
  if (n_prop == 0) return SRF_OK;
  Range rg;
  make_range(&rg, pc_range, nullptr);
  cudaStream_t st = (cudaStream_t)stream;
  SRF_COUNT(1);
  if (d.channels_last) {
    SRF_CHECK_ARG(n_cam <= IMG_MAX_CAM, "srf_img_roi_features: at most %d cameras", IMG_MAX_CAM);
    const size_t smem = (size_t)n_cam * NTAP * 8;
    if (smem > 48 * 1024) {
      SRF_CUDA(cudaFuncSetAttribute(img_roi_cl_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      SRF_CUDA(cudaFuncSetAttribute(img_roi_cl_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    if (d.channels <= 128) img_roi_cl_kernel<1><<<batch * n_prop, 256, smem, st>>>(d, boxes, n_prop, box_dim, lidar2img, n_cam, rg, o, rois_out);
    else img_roi_cl_kernel<2><<<batch * n_prop, 256, smem, st>>>(d, boxes, n_prop, box_dim, lidar2img, n_cam, rg, o, rois_out);
    SRF_LAUNCH_CHECK();
    return SRF_OK;
  }
  if (d.channels <= 128)
    img_roi_kernel<16><<<batch * n_prop, 256, 0, st>>>(d, boxes, n_prop, box_dim, lidar2img, n_cam, rg, out, channel_last, rois_out);
  else
    img_roi_kernel<32><<<batch * n_prop, 256, 0, st>>>(d, boxes, n_prop, box_dim, lidar2img, n_cam, rg, out, channel_last, rois_out);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

}  // extern "C"
