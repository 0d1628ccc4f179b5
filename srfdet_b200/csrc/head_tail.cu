// The rows of a head stage around the region-feature kernels (SURVEY.md 8f ranks 2, 3), so that the
// five cascaded stages of SRFDetHead.forward (sparse_heads/srfdet_head.py:371-458) chain on this
// library's kernels inside one CUDA graph:
//   srf_mha_attention   self-attention over the proposals (nn.MultiheadAttention core, :2281-2285)
//   srf_apply_deltas    SingleSRFDetHead.apply_deltas_lidar (:2331-2420)
//   srf_dwconv3x3_s2    DPG staircase: depthwise 3x3 stride-2 conv + BN2d + ReLU over cat(a, b) (:521-533)
//   srf_channel_sum     pfeat_34.sum(dim=1) (+ nearest resize + camera sum of the image branch, :534-595)
//   srf_gemv_f32        dpg_fc1 / dpg_fc2 on a single row per sample (:537-543)
//   srf_dpg_mix         expert softmax + weighted sum of the proposal embeddings + sigmoid of the box
//                       centres (:601-640, :403)
//   srf_decode_boxes    get_bboxes decode: sigmoid scores, denormalize_bbox, gravity -> bottom centre
//                       (:1245-1268, core/bbox/util.py:41-81)
// All fp32: these rows carry box geometry and O(P^2) softmax weights and cost microseconds.
#include "common.cuh"

namespace srf {

// ------------------------------------------------------------------------------------------------
// Self-attention core.  qkv (B*P, 3C) fp32 = in_proj(x) (q | k | v, each H heads x HD), rows batch-major.
// out (B*P, C) = softmax(q k^T / sqrt(HD)) v per (batch, head), written in any encoding (A operand of
// the out_proj GEMM).  fp32 FFMA (exact softmax weights in every precision mode).
// Block = 32 query groups x 8 key partitions; a thread owns QT queries (register tile: every K / V value read
// from shared memory feeds QT FMAs) and the keys j == part (mod 8).  K and V of the (batch, head) stream through
// shared memory in chunks, stored TRANSPOSED ([d][key]) so the 8 partitions of a warp read 8 consecutive words
// (conflict-free) and the 4 query groups of a warp share them by broadcast.  Online softmax per thread,
// partitions merged with shuffles.
// ------------------------------------------------------------------------------------------------
constexpr int ATT_QG = 32, ATT_KP = 8, ATT_CHUNK = 128;

template <int HD, int QT>
__global__ void __launch_bounds__(ATT_QG* ATT_KP) mha_attention_kernel(const float* __restrict__ qkv, int n_p, int n_heads, float scale,
                                                                       void* __restrict__ out, int out_enc) {
  __shared__ float sK[HD][ATT_CHUNK + 1];
  __shared__ float sV[HD][ATT_CHUNK + 1];
  const int C = n_heads * HD;
  const int b = blockIdx.z, h = blockIdx.y;
  const int part = threadIdx.x % ATT_KP, qg = threadIdx.x / ATT_KP;
  const int q0 = (blockIdx.x * ATT_QG + qg) * QT;
  const size_t row0 = (size_t)b * n_p;
  float q[QT][HD], acc[QT][HD], m[QT], l[QT];
#pragma unroll
  for (int t = 0; t < QT; ++t) {
    const bool live = q0 + t < n_p;
    m[t] = -INFINITY;
    l[t] = 0.f;
#pragma unroll
    for (int d = 0; d < HD; ++d) {
      q[t][d] = live ? __ldg(qkv + (row0 + q0 + t) * 3 * C + h * HD + d) * scale : 0.f;
      acc[t][d] = 0.f;
    }
  }
  for (int k0 = 0; k0 < n_p; k0 += ATT_CHUNK) {
    __syncthreads();
    for (int e = threadIdx.x; e < ATT_CHUNK * HD; e += blockDim.x) {
      const int j = e / HD, d = e % HD;                  // consecutive threads read consecutive d of one key (coalesced)
      float kv = 0.f, vv = 0.f;
      if (k0 + j < n_p) {
        const float* base = qkv + (row0 + k0 + j) * 3 * C + h * HD + d;
        kv = __ldg(base + C);
        vv = __ldg(base + 2 * C);
      }
      sK[d][j] = kv;
      sV[d][j] = vv;
    }
    __syncthreads();
    const int kn = min(ATT_CHUNK, n_p - k0);
    for (int j = part; j < kn; j += ATT_KP) {
      float s[QT];
#pragma unroll
      for (int t = 0; t < QT; ++t) s[t] = 0.f;
#pragma unroll
      for (int d = 0; d < HD; ++d) {
        const float kv = sK[d][j];
#pragma unroll
        for (int t = 0; t < QT; ++t) s[t] = fmaf(q[t][d], kv, s[t]);
      }
      float p[QT], corr[QT];
#pragma unroll
      for (int t = 0; t < QT; ++t) {
        const float mn = fmaxf(m[t], s[t]);
        corr[t] = __expf(m[t] - mn);
        p[t] = __expf(s[t] - mn);
        l[t] = l[t] * corr[t] + p[t];
        m[t] = mn;
      }
#pragma unroll
      for (int d = 0; d < HD; ++d) {
        const float vv = sV[d][j];
#pragma unroll
        for (int t = 0; t < QT; ++t) acc[t][d] = fmaf(acc[t][d], corr[t], p[t] * vv);
      }
    }
  }
#pragma unroll
  for (int t = 0; t < QT; ++t) {
    // merge the ATT_KP partitions of a query (adjacent lanes)
#pragma unroll
    for (int o = 1; o < ATT_KP; o <<= 1) {
      const float m2 = __shfl_xor_sync(0xffffffffu, m[t], o), l2 = __shfl_xor_sync(0xffffffffu, l[t], o);
      const float mn = fmaxf(m[t], m2);
      const float c1 = (m[t] == -INFINITY) ? 0.f : __expf(m[t] - mn), c2 = (m2 == -INFINITY) ? 0.f : __expf(m2 - mn);
      l[t] = l[t] * c1 + l2 * c2;
#pragma unroll
      for (int d = 0; d < HD; ++d) acc[t][d] = acc[t][d] * c1 + __shfl_xor_sync(0xffffffffu, acc[t][d], o) * c2;
      m[t] = mn;
    }
    if (q0 + t < n_p && part == 0) {
      const float inv = 1.f / l[t];
      const size_t row = row0 + q0 + t;
      if (out_enc == SRF_F32) {
        float* o = (float*)out + row * C + h * HD;
#pragma unroll
        for (int d = 0; d < HD; ++d) o[d] = acc[t][d] * inv;
      } else {
        const bool f16 = enc_is_f16(out_enc), split = enc_is_split(out_enc);
        uint16_t* o = (uint16_t*)out + row * C * (split ? 2 : 1) + h * HD;
#pragma unroll
        for (int d = 0; d < HD; d += 2) {
          uint32_t hi, lo;
          split16x2(f16, acc[t][d] * inv, acc[t][d + 1] * inv, hi, lo);
          *reinterpret_cast<uint32_t*>(o + d) = hi;
          if (split) *reinterpret_cast<uint32_t*>(o + C + d) = lo;
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
__global__ void apply_deltas_kernel(const float* __restrict__ deltas, const float* __restrict__ boxes, int k, int dim,
                                    const float* __restrict__ wts, float scale_clamp, float lo0, float lo1, float lo2, float sp0, float sp1,
                                    float sp2, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= k) return;
  const float* d = deltas + (size_t)i * dim;
  const float* bx = boxes + (size_t)i * dim;
  float* o = out + (size_t)i * dim;
  const float lo[3] = {lo0, lo1, lo2}, sp[3] = {sp0, sp1, sp2};
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const float size = expf(bx[3 + j]);                               // boxes carry log sizes
    const float dxyz = d[j] / __ldg(wts + j);
    const float dwlh = fminf(d[3 + j] / __ldg(wts + 3 + j), scale_clamp);
    const float ctr = dxyz * size + bx[j];                            // absolute centre (after the in-place de-normalisation)
    o[j] = fminf(fmaxf((ctr - lo[j]) / sp[j], 0.f), 1.f);             // back to [0,1]
    o[3 + j] = logf(expf(dwlh) * size);
  }
  for (int j = 6; j < dim; ++j) o[j] = d[j];                          // sin, cos (, vx, vy): raw deltas
}

// ------------------------------------------------------------------------------------------------
// DPG staircase.  A map is (n, C, H, W) addressed through element strides (sn, sc, sh, sw), so both
// NCHW and torch.channels_last tensors are read in place.
struct MapView {
  const float* p;
  int c;
  long long sn, sc, sh, sw;
};

// out = relu(bn(dwconv3x3_s2_p1(cat(a, b)))); w (Ca+Cb, 9) with BN folded, bias (Ca+Cb).  out is
// (n, Ca+Cb, Ho, Wo) NCHW, or (n, Ho, Wo, Ca+Cb) when cl_out (channel-fastest threads: coalesced on
// torch.channels_last inputs)
// channels_last fast path: a thread owns 4 consecutive channels (float4 loads / stores; a.c and b.c multiples of 4) of
// DW_PX consecutive output pixels of a row.  The folded weights sit in shared memory transposed to [tap][channel] (one
// conflict-free LDS.128 per tap instead of 36 registers per thread: 4 blocks of 256 threads per SM keep ~80 KB of loads in
// flight, the kernel streams its input once from HBM); per kernel row the 2*DW_PX+1 input columns are loaded as one batch
// and shared by the DW_PX outputs.  Index math is 32-bit.
constexpr int DW_PX = 2;
__global__ void __launch_bounds__(256, 4) dwconv3x3_s2_cl4_kernel(MapView a, MapView b, int n, int h, int w, int ho, int wo,
                                                                  const float* __restrict__ wt, const float* __restrict__ bias, int relu,
                                                                  float* __restrict__ out) {
  extern __shared__ __align__(16) float dw_smem[];     // [9][ctot] weights, [ctot] bias
  const int ctot = a.c + b.c, c4n = ctot / 4;
  for (int i = threadIdx.x; i < ctot * 9; i += blockDim.x) dw_smem[(i % 9) * ctot + i / 9] = __ldg(wt + i);
  for (int i = threadIdx.x; i < ctot; i += blockDim.x) dw_smem[9 * ctot + i] = __ldg(bias + i);
  __syncthreads();
  const int wq = (wo + DW_PX - 1) / DW_PX;
  const unsigned total = (unsigned)n * ho * wq * c4n;
  for (unsigned e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    const int c = (int)(e % c4n) * 4;
    unsigned t = e / c4n;
    const int xq = (int)(t % wq);
    t /= wq;
    const int y = (int)(t % ho), img = (int)(t / ho);
    const MapView& mv = c < a.c ? a : b;
    const int cl = c < a.c ? c : c - a.c;
    const float* base = mv.p + (long long)img * mv.sn + cl;          // sc == 1
    const float4 bz = *reinterpret_cast<const float4*>(dw_smem + 9 * ctot + c);
    float4 acc[DW_PX];
#pragma unroll
    for (int px = 0; px < DW_PX; ++px) acc[px] = bz;
    const int x0 = xq * DW_PX * 2 - 1;                               // first input column of the patch
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const int iy = 2 * y - 1 + ky;
      if (iy < 0 || iy >= h) continue;
      const float* rowp = base + (long long)iy * mv.sh;
      float4 v[2 * DW_PX + 1];
#pragma unroll
      for (int j = 0; j < 2 * DW_PX + 1; ++j) {
        const int ix = x0 + j;
        v[j] = (ix >= 0 && ix < w) ? __ldg(reinterpret_cast<const float4*>(rowp + (long long)ix * mv.sw)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const float4 wv = *reinterpret_cast<const float4*>(dw_smem + (ky * 3 + kx) * ctot + c);
#pragma unroll
        for (int px = 0; px < DW_PX; ++px) {
          const float4 u = v[2 * px + kx];
          acc[px].x = fmaf(u.x, wv.x, acc[px].x);
          acc[px].y = fmaf(u.y, wv.y, acc[px].y);
          acc[px].z = fmaf(u.z, wv.z, acc[px].z);
          acc[px].w = fmaf(u.w, wv.w, acc[px].w);
        }
      }
    }
#pragma unroll
    for (int px = 0; px < DW_PX; ++px) {
      const int x = xq * DW_PX + px;
      if (x >= wo) break;
      float4 r = acc[px];
      if (relu) { r.x = fmaxf(r.x, 0.f); r.y = fmaxf(r.y, 0.f); r.z = fmaxf(r.z, 0.f); r.w = fmaxf(r.w, 0.f); }
      *reinterpret_cast<float4*>(out + (((size_t)img * ho + y) * wo + x) * ctot + c) = r;
    }
  }
}

__global__ void dwconv3x3_s2_kernel(MapView a, MapView b, int n, int h, int w, int ho, int wo, const float* __restrict__ wt,
                                    const float* __restrict__ bias, int relu, int cl_out, float* __restrict__ out) {
  const int ctot = a.c + b.c;
  const long long total = (long long)n * ctot * ho * wo;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    int x, y, c, img;
    if (cl_out) {
      c = (int)(e % ctot);
      long long t = e / ctot;
      x = (int)(t % wo);
      t /= wo;
      y = (int)(t % ho);
      img = (int)(t / ho);
    } else {
      x = (int)(e % wo);
      long long t = e / wo;
      y = (int)(t % ho);
      t /= ho;
      c = (int)(t % ctot);
      img = (int)(t / ctot);
    }
    const MapView& mv = c < a.c ? a : b;
    const int cl = c < a.c ? c : c - a.c;
    const float* base = mv.p + img * mv.sn + cl * mv.sc;
    float acc = __ldg(bias + c);
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const int iy = 2 * y - 1 + ky;
      if (iy < 0 || iy >= h) continue;
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const int ix = 2 * x - 1 + kx;
        if (ix < 0 || ix >= w) continue;
        acc = fmaf(__ldg(base + iy * mv.sh + ix * mv.sw), __ldg(wt + c * 9 + ky * 3 + kx), acc);
      }
    }
    out[e] = relu ? fmaxf(acc, 0.f) : acc;
  }
}

// out[s, oy*wo + ox] = sum over the `group` images of sample s and over the channels of cat(a, b) at the
// nearest source pixel (F.interpolate(mode='nearest') index: floor(o * in / out)); group = 1 and
// (ho, wo) = (h, w) is the plain channel sum of the LiDAR branch.
__global__ void channel_sum_kernel(MapView a, MapView b, int n_samples, int group, int h, int w, int ho, int wo, float* __restrict__ out) {
  const int o = blockIdx.x, s = blockIdx.y;
  const int oy = o / wo, ox = o % wo;
  const int iy = min((int)floorf((float)oy * ((float)h / (float)ho)), h - 1);
  const int ix = min((int)floorf((float)ox * ((float)w / (float)wo)), w - 1);
  const int ctot = a.c + b.c;
  float acc = 0.f;
  for (int e = threadIdx.x; e < group * ctot; e += blockDim.x) {
    const int g = e / ctot, c = e % ctot;
    const MapView& mv = c < a.c ? a : b;
    const int cl = c < a.c ? c : c - a.c;
    acc += __ldg(mv.p + (long long)(s * group + g) * mv.sn + cl * mv.sc + iy * mv.sh + ix * mv.sw);
  }
  __shared__ float red[32];
  for (int off = 16; off; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += red[i];
    out[(size_t)s * ho * wo + o] = t;
  }
}

// out (m, n) = act(x (m, k) . W (n, k)^T + bias): one warp per output column, GEMV_MAXM rows of x at once; blockIdx.y
// picks the group of rows [8y, 8y + 8).  A row's sum does not depend on the other rows of its group or on the group, so
// every row comes out as it does in a call of that row alone.
constexpr int GEMV_MAXM = 8;
__global__ void __launch_bounds__(256) gemv_kernel(const float* __restrict__ x, int m, int k, const float* __restrict__ w, int n,
                                                   const float* __restrict__ bias, int relu, float* __restrict__ out) {
  const int col = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (col >= n) return;
  const int r0 = blockIdx.y * GEMV_MAXM;
  x += (size_t)r0 * k;
  out += (size_t)r0 * n;
  m = min(m - r0, GEMV_MAXM);
  float acc[GEMV_MAXM];
#pragma unroll
  for (int r = 0; r < GEMV_MAXM; ++r) acc[r] = 0.f;
  const float* wr = w + (size_t)col * k;
  for (int j = lane; j < k; j += 32) {
    const float wv = __ldg(wr + j);
#pragma unroll
    for (int r = 0; r < GEMV_MAXM; ++r)
      if (r < m) acc[r] = fmaf(__ldg(x + (size_t)r * k + j), wv, acc[r]);
  }
#pragma unroll
  for (int r = 0; r < GEMV_MAXM; ++r) {
    if (r >= m) break;
    float v = acc[r];
    for (int off = 16; off; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    if (lane == 0) {
      v += bias ? __ldg(bias + col) : 0.f;
      out[(size_t)r * n + col] = relu ? fmaxf(v, 0.f) : v;
    }
  }
}

// logits_a (+ logits_b)/2 -> softmax over the E experts -> boxes (B,P,D) = sum_e w * emb_boxes[e,p,:]
// with sigmoid on the first three (centre) coordinates, feats (B,P,C) = sum_e w * emb_feats[e,p,:]
__global__ void dpg_mix_kernel(const float* __restrict__ la, const float* __restrict__ lb, int n_b, int n_e, int n_p,
                               const float* __restrict__ emb_boxes, int dim, const float* __restrict__ emb_feats, int c,
                               float* __restrict__ boxes, float* __restrict__ feats, int sigmoid_centres) {
  const int p = blockIdx.x, b = blockIdx.y;
  __shared__ float wgt[16];
  if (threadIdx.x == 0) {
    float mx = -INFINITY;
    for (int e = 0; e < n_e; ++e) {
      float v = la[((size_t)b * n_e + e) * n_p + p];
      if (lb) v = (v + lb[((size_t)b * n_e + e) * n_p + p]) / 2.f;
      wgt[e] = v;
      mx = fmaxf(mx, v);
    }
    float s = 0.f;
    for (int e = 0; e < n_e; ++e) { wgt[e] = expf(wgt[e] - mx); s += wgt[e]; }
    for (int e = 0; e < n_e; ++e) wgt[e] /= s;
  }
  __syncthreads();
  for (int j = threadIdx.x; j < dim + c; j += blockDim.x) {
    float acc = 0.f;
    if (j < dim) {
      for (int e = 0; e < n_e; ++e) acc += wgt[e] * __ldg(emb_boxes + ((size_t)e * n_p + p) * dim + j);
      if (j < 3 && sigmoid_centres) acc = 1.f / (1.f + expf(-acc));
      boxes[((size_t)b * n_p + p) * dim + j] = acc;
    } else {
      const int cc = j - dim;
      for (int e = 0; e < n_e; ++e) acc += wgt[e] * __ldg(emb_feats + ((size_t)e * n_p + p) * c + cc);
      feats[((size_t)b * n_p + p) * c + cc] = acc;
    }
  }
}

// scores = sigmoid(logits); boxes (k, dim) [cx,cy,cz (absolute), log w,l,h, sin, cos (, vx, vy)] ->
// (k, dim-1) [cx, cy, cz - h/2, w, l, h, atan2(sin, cos) (, vx, vy)]
__global__ void decode_boxes_kernel(const float* __restrict__ logits, long long n_logits, const float* __restrict__ boxes, int k, int dim,
                                    float* __restrict__ scores, float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_logits) scores[i] = 1.f / (1.f + expf(-logits[i]));
  if (i < k) {
    const float* b = boxes + i * dim;
    float* o = out + i * (dim - 1);
    const float hgt = expf(b[5]);
    o[0] = b[0]; o[1] = b[1]; o[2] = b[2] - hgt * 0.5f;
    o[3] = expf(b[3]); o[4] = expf(b[4]); o[5] = hgt;
    o[6] = atan2f(b[6], b[7]);
    for (int j = 8; j < dim; ++j) o[j - 1] = b[j];
  }
}

static int egrid(long long n, int threads) {
  long long g = (n + threads - 1) / threads;
  const long long cap = (long long)sm_count() * 16;
  if (g > cap) g = cap;
  return g < 1 ? 1 : (int)g;
}

static MapView make_view(const srf_map* m) {
  MapView v;
  v.p = m ? m->ptr : nullptr;
  v.c = (m && m->ptr) ? m->c : 0;
  v.sn = m ? m->sn : 0; v.sc = m ? m->sc : 0; v.sh = m ? m->sh : 0; v.sw = m ? m->sw : 0;
  return v;
}

}  // namespace srf

using namespace srf;

extern "C" {

int srf_mha_attention(const float* qkv, int32_t n_batch, int32_t n_p, int32_t n_heads, int32_t head_dim, void* out, int32_t out_enc,
                      void* stream) {
  SRF_CHECK_ARG(qkv && out && n_batch >= 1 && n_p >= 0 && n_heads >= 1, "srf_mha_attention: bad args");
  SRF_CHECK_ARG(out_enc == SRF_F32 || enc_is_16(out_enc), "srf_mha_attention: bad output encoding");
  if (n_p == 0) return SRF_OK;
  const float scale = 1.f / sqrtf((float)head_dim);
  cudaStream_t st = (cudaStream_t)stream;
  SRF_COUNT(1);
  // 16-bit modes: tensor-core kernel (attention.cu); fp32 / split outputs: the fp32 kernel below
  if (mha_attention_mma_launch(qkv, n_batch, n_p, n_heads, head_dim, out, out_enc, st)) {
    SRF_LAUNCH_CHECK();
    return SRF_OK;
  }
  constexpr int T = ATT_QG * ATT_KP;
  switch (head_dim) {     // QT queries per thread: 2 (64 queries per block: 120 blocks for 900 proposals x 8 heads), 1 for 32-wide heads
    case 8: mha_attention_kernel<8, 2><<<dim3(cdiv(n_p, ATT_QG * 2), n_heads, n_batch), T, 0, st>>>(qkv, n_p, n_heads, scale, out, out_enc); break;
    case 16: mha_attention_kernel<16, 2><<<dim3(cdiv(n_p, ATT_QG * 2), n_heads, n_batch), T, 0, st>>>(qkv, n_p, n_heads, scale, out, out_enc); break;
    case 32: mha_attention_kernel<32, 1><<<dim3(cdiv(n_p, ATT_QG), n_heads, n_batch), T, 0, st>>>(qkv, n_p, n_heads, scale, out, out_enc); break;
    default: set_error("srf_mha_attention: head_dim must be 8/16/32 (got %d)", head_dim); return SRF_ERR_UNSUPPORTED;
  }
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

int srf_apply_deltas(const float* deltas, const float* boxes, int32_t k, int32_t dim, const float* weights, float scale_clamp,
                     const float pc_range[6], float* out, void* stream) {
  SRF_CHECK_ARG(deltas && boxes && weights && pc_range && out && k >= 0 && dim >= 8, "srf_apply_deltas: bad args");
  if (k == 0) return SRF_OK;
  SRF_COUNT(1);
  apply_deltas_kernel<<<cdiv(k, 128), 128, 0, (cudaStream_t)stream>>>(deltas, boxes, k, dim, weights, scale_clamp, pc_range[0], pc_range[1],
                                                                     pc_range[2], pc_range[3] - pc_range[0], pc_range[4] - pc_range[1],
                                                                     pc_range[5] - pc_range[2], out);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

int srf_dwconv3x3_s2(const srf_map* a, const srf_map* b, int32_t n, int32_t h, int32_t w, const float* wt_folded, const float* bias_folded,
                     int32_t relu, int32_t channels_last_out, float* out, void* stream) {
  SRF_CHECK_ARG(a && a->ptr && wt_folded && bias_folded && out && n >= 1 && h >= 1 && w >= 1, "srf_dwconv3x3_s2: bad args");
  const MapView va = make_view(a), vb = make_view(b);
  const int ho = (h + 2 - 3) / 2 + 1, wo = (w + 2 - 3) / 2 + 1;
  const long long total = (long long)n * (va.c + vb.c) * ho * wo;
  SRF_COUNT(1);
  const bool vec = channels_last_out && total < (1ll << 31) && va.c + vb.c <= 1024 && va.sc == 1 && (vb.c == 0 || vb.sc == 1) && va.c % 4 == 0 && vb.c % 4 == 0 &&
                   va.sw % 4 == 0 && va.sh % 4 == 0 && va.sn % 4 == 0 && (vb.c == 0 || (vb.sw % 4 == 0 && vb.sh % 4 == 0 && vb.sn % 4 == 0)) &&
                   ((uintptr_t)va.p % 16 == 0) && (vb.c == 0 || (uintptr_t)vb.p % 16 == 0);
  if (vec) {
    const long long nthr = (long long)n * ho * ((wo + DW_PX - 1) / DW_PX) * ((va.c + vb.c) / 4);
    dwconv3x3_s2_cl4_kernel<<<egrid(nthr, 256), 256, (size_t)(va.c + vb.c) * 10 * sizeof(float), (cudaStream_t)stream>>>(va, vb, n, h, w, ho, wo, wt_folded, bias_folded, relu, out);
    SRF_LAUNCH_CHECK();
    return SRF_OK;
  }
  dwconv3x3_s2_kernel<<<egrid(total, 256), 256, 0, (cudaStream_t)stream>>>(va, vb, n, h, w, ho, wo, wt_folded, bias_folded, relu, channels_last_out, out);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

int srf_channel_sum(const srf_map* a, const srf_map* b, int32_t n_samples, int32_t group, int32_t h, int32_t w, int32_t ho, int32_t wo,
                    float* out, void* stream) {
  SRF_CHECK_ARG(a && a->ptr && out && n_samples >= 1 && group >= 1 && h >= 1 && w >= 1 && ho >= 1 && wo >= 1, "srf_channel_sum: bad args");
  const MapView va = make_view(a), vb = make_view(b);
  SRF_COUNT(1);
  channel_sum_kernel<<<dim3(ho * wo, n_samples), 128, 0, (cudaStream_t)stream>>>(va, vb, n_samples, group, h, w, ho, wo, out);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

int srf_gemv_f32(const float* x, int32_t m, int32_t k, const float* w, int32_t n, const float* bias, int32_t relu, float* out,
                 void* stream) {
  SRF_CHECK_ARG(x && w && out && m >= 1 && m <= 65535 * GEMV_MAXM && k >= 1 && n >= 1, "srf_gemv_f32: need 1 <= m <= %d rows",
                65535 * GEMV_MAXM);
  SRF_COUNT(1);
  gemv_kernel<<<dim3(cdiv(n, 8), cdiv(m, GEMV_MAXM)), 256, 0, (cudaStream_t)stream>>>(x, m, k, w, n, bias, relu, out);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

int srf_dpg_mix(const float* logits_a, const float* logits_b, int32_t n_batch, int32_t n_exp, int32_t n_p, const float* emb_boxes,
                int32_t box_dim, const float* emb_feats, int32_t c, float* boxes, float* feats, int32_t sigmoid_centres, void* stream) {
  SRF_CHECK_ARG(logits_a && emb_boxes && emb_feats && boxes && feats && n_batch >= 1 && n_exp >= 1 && n_exp <= 16 && n_p >= 1,
                "srf_dpg_mix: bad args (at most 16 experts)");
  SRF_COUNT(1);
  dpg_mix_kernel<<<dim3(n_p, n_batch), 128, 0, (cudaStream_t)stream>>>(logits_a, logits_b, n_batch, n_exp, n_p, emb_boxes, box_dim, emb_feats,
                                                                      c, boxes, feats, sigmoid_centres);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

int srf_decode_boxes(const float* logits, int64_t n_logits, const float* boxes, int32_t k, int32_t dim, float* scores, float* out,
                     void* stream) {
  SRF_CHECK_ARG(logits && boxes && scores && out && k >= 0 && dim >= 8 && n_logits >= 0, "srf_decode_boxes: bad args");
  const long long n = n_logits > k ? n_logits : k;
  if (n == 0) return SRF_OK;
  SRF_COUNT(1);
  decode_boxes_kernel<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(logits, n_logits, boxes, k, dim, scores, out);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

}  // extern "C"
