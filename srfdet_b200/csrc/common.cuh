// Shared helpers for the sm_100a kernels of libsrfdet_b200.so.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "../../include/srfdet_b200.h"

namespace srf {

void set_error(const char* fmt, ...);
extern unsigned long long g_launches;  // kernels launched by this library (bench evidence)
#define SRF_COUNT(n) (srf::g_launches += (n))
int sm_count();
int spconv16_warp_launch(const srf_conv_args* cv, bool f16, cudaStream_t st);   // spconv_warp16.cu
bool mha_attention_mma_launch(const float* qkv, int n_batch, int n_p, int n_heads, int head_dim, void* out, int out_enc, cudaStream_t st);   // attention.cu

#define SRF_CHECK_ARG(cond, ...)          \
  do {                                    \
    if (!(cond)) {                        \
      srf::set_error(__VA_ARGS__);        \
      return SRF_ERR_ARG;                 \
    }                                     \
  } while (0)

#define SRF_CUDA(expr)                                                                  \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess) {                                                            \
      srf::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__,  \
                     __LINE__);                                                         \
      return SRF_ERR_CUDA;                                                              \
    }                                                                                   \
  } while (0)

#define SRF_LAUNCH_CHECK() SRF_CUDA(cudaGetLastError())

static inline int cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// ------------------------------------------------------------------------------------
// Cell index (occupancy bitmap + per-word exclusive rank).  Layout inside the caller's
// buffer:  [bits: nwords u32][rank: nwords u32][blocksum: SCAN_BLOCKS u32]
// ------------------------------------------------------------------------------------
constexpr int SCAN_BLOCKS = 1024;
constexpr int SCAN_THREADS = 256;

struct IndexView {
  uint32_t* bits;
  uint32_t* rank;
  uint32_t* blocksum;
  int64_t nwords;
};

static inline int64_t index_nwords(int64_t ncells) { return (ncells + 31) / 32; }

static inline IndexView index_view(const void* p, int64_t ncells) {
  IndexView v;
  v.nwords = index_nwords(ncells);
  int64_t nw_al = (v.nwords + 3) / 4 * 4;
  v.bits = (uint32_t*)p;
  v.rank = v.bits + nw_al;
  v.blocksum = v.rank + nw_al;
  return v;
}

struct Dims4 {
  int32_t b, z, y, x;
};

__device__ __forceinline__ int64_t cell_of(const Dims4& d, int b, int z, int y, int x) {
  return (((int64_t)b * d.z + z) * d.y + y) * d.x + x;
}

// rank of an occupied cell, or -1
__device__ __forceinline__ int index_rank(const uint32_t* __restrict__ bits,
                                          const uint32_t* __restrict__ rank, int64_t cell) {
  int64_t w = cell >> 5;
  uint32_t bit = 1u << (cell & 31);
  uint32_t word = __ldg(bits + w);
  if (!(word & bit)) return -1;
  return (int)(__ldg(rank + w) + __popc(word & (bit - 1)));
}

// device-wide exclusive scan of uint32 values produced by a functor; 3 launches.
// (implemented in index.cu; used by voxelize.cu as well)
int scan_flags_launch(const uint32_t* in, uint32_t* out_excl, uint32_t* blocksum, int64_t n,
                      int32_t* d_total, int popcount_mode, cudaStream_t st);

__device__ __forceinline__ float bf16_bits_to_float(uint32_t hi16) { return __uint_as_float(hi16 << 16); }

// ------------------------------------------------------------------------------------
// 16-bit element encodings (include/srfdet_b200.h: SRF_BF16 / SRF_F16 and the split forms
// SRF_BF16X2 / SRF_F16X2 = [hi | lo] rows with value = hi + lo).
// ------------------------------------------------------------------------------------
static inline __host__ __device__ bool enc_is_split(int e) { return e == SRF_BF16X2 || e == SRF_F16X2; }
static inline __host__ __device__ bool enc_is_f16(int e) { return e == SRF_F16 || e == SRF_F16X2; }
static inline __host__ __device__ bool enc_is_16(int e) { return e >= SRF_BF16 && e <= SRF_F16X2; }
// bytes of one row of c values
static inline __host__ __device__ int enc_row_bytes(int e, int c) { return e == SRF_F32 ? 4 * c : (enc_is_split(e) ? 4 * c : 2 * c); }

// two fp32 values -> one 32-bit word of two 16-bit elements (low half = a); f16 saturates at +-65504
__device__ __forceinline__ uint32_t pack16x2(bool f16, float a, float b) {
  if (f16) {
    a = fminf(fmaxf(a, -65504.f), 65504.f);
    b = fminf(fmaxf(b, -65504.f), 65504.f);
    const __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&h);
  }
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ float2 unpack16x2(bool f16, uint32_t w) {
  if (f16) return __half22float2(*reinterpret_cast<const __half2*>(&w));
  return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
}
__device__ __forceinline__ uint16_t pack16(bool f16, float a) { return (uint16_t)(pack16x2(f16, a, 0.f) & 0xffffu); }
__device__ __forceinline__ float unpack16(bool f16, uint16_t h) { return unpack16x2(f16, (uint32_t)h).x; }
// split a pair: hi word and lo word (lo = round16(v - hi))
__device__ __forceinline__ void split16x2(bool f16, float a, float b, uint32_t& hi, uint32_t& lo) {
  hi = pack16x2(f16, a, b);
  const float2 h = unpack16x2(f16, hi);
  lo = pack16x2(f16, a - h.x, b - h.y);
}

// Row encoder of srf_nchw_to_rows and srf_pillar_encode_rows: stores channel ch (value v0) and channel ch + 1 (v1, when
// ch + 1 < c) of one row of c values in encoding enc.  ch is even.  SRF_F32 rows are plain; the 16-bit forms store the
// pair as one 32-bit word (hi, then lo for the split forms) when c is even, element by element otherwise.
__device__ __forceinline__ void store_row_pair(int enc, void* row, int c, int ch, float v0, float v1) {
  if (enc == SRF_F32) {
    float* r = static_cast<float*>(row);
    r[ch] = v0;
    if (ch + 1 < c) r[ch + 1] = v1;
    return;
  }
  const bool f16 = enc_is_f16(enc), split = enc_is_split(enc);
  uint16_t* r = static_cast<uint16_t*>(row);
  if (ch + 1 < c && (c & 1) == 0) {
    uint32_t h, l;
    split16x2(f16, v0, v1, h, l);
    *reinterpret_cast<uint32_t*>(r + ch) = h;
    if (split) *reinterpret_cast<uint32_t*>(r + c + ch) = l;
  } else {
    const uint16_t h0 = pack16(f16, v0);
    r[ch] = h0;
    if (split) r[c + ch] = pack16(f16, v0 - unpack16(f16, h0));
    if (ch + 1 < c) {
      const uint16_t h1 = pack16(f16, v1);
      r[ch + 1] = h1;
      if (split) r[c + ch + 1] = pack16(f16, v1 - unpack16(f16, h1));
    }
  }
}


// ---------------------------------------------------------------------------------------
// Programmatic dependent launch: a kernel launched through launch_pdl() may be scheduled while
// its predecessor on the stream is still draining (its launch latency and prologue overlap
// the predecessor's tail).  Such a kernel MUST execute pdl_wait() before it touches anything
// the predecessor wrote; pdl_trigger() lets the successor start launching.  Both are no-ops
// for plain launches.  SRFDET_B200_PDL=0 falls back to plain launches.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

static inline bool pdl_enabled() {
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("SRFDET_B200_PDL");
    on = (e && e[0] == '0') ? 0 : 1;
  }
  return on != 0;
}

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

}  // namespace srf
