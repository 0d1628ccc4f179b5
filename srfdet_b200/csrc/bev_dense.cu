// Helpers of the dense BEV backbone / neck (SURVEY.md 8f rank 1: SECONDCustom
// models/backbones/second_custom.py:23-91 + mmdet FPN).  The convolutions themselves run on the
// gather-GEMM kernel (igemm_umma.cu) over NHWC pixel rows with a dense rulebook (index.cu); this file
// has the two layout / elementwise steps around them:
//   srf_nchw_to_rows   (n, c, h, w) fp32 NCHW (SparseConvTensor.dense() layout) -> (n*h*w, c) rows in a
//                      16-bit encoding (the A operand of the first backbone conv)
//   srf_upsample_add   FPN top-down step: rows_hi += nearest_upsample(rows_lo)  (mmdet fpn.py, F.interpolate
//                      mode='nearest' with size=)
#include "common.cuh"

namespace srf {

// tile transpose through shared memory: 64 channels x 32 pixels per CTA; coalesced 128-byte reads along w, and 128-byte
// writes along c (a lane packs two adjacent channels into one 32-bit store)
__global__ void __launch_bounds__(256) nchw_to_rows_kernel(const float* __restrict__ in, int c, int hw, int enc, uint16_t* __restrict__ out) {
  __shared__ float tile[64][33];
  const int img = blockIdx.z;
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 64;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;     // 32 x 8
  const float* src = in + (size_t)img * c * hw;
#pragma unroll
  for (int j = ty; j < 64; j += 8) {
    const int ch = c0 + j, p = p0 + tx;
    tile[j][tx] = (ch < c && p < hw) ? __ldg(src + (size_t)ch * hw + p) : 0.f;
  }
  __syncthreads();
  const int width = enc_is_split(enc) ? 2 * c : c;
  const int ch = c0 + 2 * tx;
#pragma unroll
  for (int j = ty; j < 32; j += 8) {
    const int p = p0 + j;
    if (p >= hw || ch >= c) continue;
    store_row_pair(enc, out + ((size_t)img * hw + p) * width, c, ch, tile[2 * tx][j], tile[2 * tx + 1][j]);
  }
}

// hi (n, h, w, c) rows, lo (n, hl, wl, c) rows, both in encoding enc; hi += lo[nearest]
__global__ void upsample_add_kernel(uint16_t* __restrict__ hi, const uint16_t* __restrict__ lo, int n, int h, int w, int hl, int wl, int c,
                                    int enc) {
  const bool f16 = enc_is_f16(enc), split = enc_is_split(enc);
  const int width = split ? 2 * c : c;
  const int64_t total = (int64_t)n * h * w * (c / 2);
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int cp = (int)(e % (c / 2)) * 2;
    int64_t t = e / (c / 2);
    const int x = (int)(t % w);
    t /= w;
    const int y = (int)(t % h), img = (int)(t / h);
    const int ys = min((int)floorf((float)y * ((float)hl / (float)h)), hl - 1);
    const int xs = min((int)floorf((float)x * ((float)wl / (float)w)), wl - 1);
    uint16_t* ph = hi + (((size_t)img * h + y) * w + x) * width + cp;
    const uint16_t* pl = lo + (((size_t)img * hl + ys) * wl + xs) * width + cp;
    float2 a = unpack16x2(f16, *reinterpret_cast<const uint32_t*>(ph));
    float2 b = unpack16x2(f16, *reinterpret_cast<const uint32_t*>(pl));
    if (split) {
      const float2 a2 = unpack16x2(f16, *reinterpret_cast<const uint32_t*>(ph + c));
      const float2 b2 = unpack16x2(f16, *reinterpret_cast<const uint32_t*>(pl + c));
      a.x += a2.x; a.y += a2.y; b.x += b2.x; b.y += b2.y;
    }
    uint32_t oh, ol;
    split16x2(f16, a.x + b.x, a.y + b.y, oh, ol);
    *reinterpret_cast<uint32_t*>(ph) = oh;
    if (split) *reinterpret_cast<uint32_t*>(ph + c) = ol;
  }
}

}  // namespace srf

using namespace srf;

extern "C" {

int srf_nchw_to_rows(const float* in, int32_t n, int32_t c, int32_t h, int32_t w, int32_t enc, void* out, void* stream) {
  SRF_CHECK_ARG(in && out && n >= 1 && c >= 1 && h >= 1 && w >= 1 && enc_is_16(enc), "srf_nchw_to_rows: bad args");
  dim3 grid(cdiv((int64_t)h * w, 32), cdiv(c, 64), n);
  SRF_COUNT(1);
  nchw_to_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(in, c, h * w, enc, (uint16_t*)out);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

int srf_upsample_add(void* rows_hi, const void* rows_lo, int32_t n, int32_t h, int32_t w, int32_t h_lo, int32_t w_lo, int32_t c,
                     int32_t enc, void* stream) {
  SRF_CHECK_ARG(rows_hi && rows_lo && n >= 1 && h >= 1 && w >= 1 && h_lo >= 1 && w_lo >= 1 && c >= 2 && c % 2 == 0 && enc_is_16(enc),
                "srf_upsample_add: bad args");
  int64_t total = (int64_t)n * h * w * (c / 2);
  int64_t g = (total + 255) / 256;
  if (g > sm_count() * 16) g = sm_count() * 16;
  SRF_COUNT(1);
  upsample_add_kernel<<<(int)g, 256, 0, (cudaStream_t)stream>>>((uint16_t*)rows_hi, (const uint16_t*)rows_lo, n, h, w, h_lo, w_lo, c, enc);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

}  // extern "C"
