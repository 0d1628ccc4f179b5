// FP32 ("exact") sparse convolution and linear kernels on the SIMT pipes, plus the
// weight-packing / conversion helpers used by the tcgen05 path.
//
// The FP32 kernels are the parity mode (tolerance 1e-4 vs the fp32 reference): same
// output-stationary rulebook as the tensor-core kernel, FFMA accumulation in fp32.
#include <stdlib.h>

#include "common.cuh"

namespace srf {

// one value of a row-major (rows, c) buffer in encoding `enc` (split rows are [hi(c) | lo(c)])
__device__ __forceinline__ float ld_enc(const void* p, int enc, size_t row, int c, int col) {
  if (enc == SRF_F32) return __ldg((const float*)p + row * c + col);
  const bool f16 = enc_is_f16(enc);
  const uint16_t* q = (const uint16_t*)p;
  if (!enc_is_split(enc)) return unpack16(f16, q[row * c + col]);
  return unpack16(f16, q[row * 2 * c + col]) + unpack16(f16, q[row * 2 * c + c + col]);
}
__device__ __forceinline__ void st_enc(void* p, int enc, size_t row, int c, int col, float v) {
  if (enc == SRF_F32) { ((float*)p)[row * c + col] = v; return; }
  const bool f16 = enc_is_f16(enc);
  uint16_t* q = (uint16_t*)p;
  if (!enc_is_split(enc)) { q[row * c + col] = pack16(f16, v); return; }
  const uint16_t h = pack16(f16, v);
  q[row * 2 * c + col] = h;
  q[row * 2 * c + c + col] = pack16(f16, v - unpack16(f16, h));
}

template <typename T>
__device__ __forceinline__ float ld_as_float(const T* p);
template <>
__device__ __forceinline__ float ld_as_float<float>(const float* p) { return __ldg(p); }
template <>
__device__ __forceinline__ float ld_as_float<__nv_bfloat16>(const __nv_bfloat16* p) {
  return __bfloat162float(*p);
}

struct ConvDev {
  const void* in;
  const int32_t* nbr;
  const uint32_t* tile_mask;
  const int32_t* d_n_out;
  const float* w;
  const float* bias;
  const void* residual;
  void* out;
  float* dense;
  const int4* out_coors;
  int cin, kvol, cap_out, relu, out_enc;
  int D, H, W;
};

constexpr int SIMT_TILE = 32;
constexpr int SIMT_MAXCIN = 128;

// block = 128 threads, tile = 32 output rows.  thread -> one output channel `co` and
// RPT = COUT/4 rows; A tile (32 x cin) staged in shared memory, weights read through L1.
template <int COUT, typename TIN>
__global__ void __launch_bounds__(128) spconv_f32_kernel(ConvDev a) {
  constexpr int NGROUPS = 128 / COUT;
  constexpr int RPT = SIMT_TILE / NGROUPS;
  __shared__ float sA[SIMT_TILE][SIMT_MAXCIN + 1];
  __shared__ int sN[SIMT_TILE];
  const int n_out = a.d_n_out ? min(*a.d_n_out, a.cap_out) : a.cap_out;
  const int ntiles = (n_out + SIMT_TILE - 1) / SIMT_TILE;
  const int co = threadIdx.x % COUT;
  const int rg = threadIdx.x / COUT;
  const TIN* in = (const TIN*)a.in;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int row0 = tile * SIMT_TILE;
    float acc[RPT];
#pragma unroll
    for (int r = 0; r < RPT; ++r) acc[r] = 0.f;
    const uint32_t mask = a.tile_mask ? a.tile_mask[row0 >> 7] : 0xffffffffu;
    for (int k = 0; k < a.kvol; ++k) {
      if (!((mask >> k) & 1u)) continue;
      int nb = -1;
      if (threadIdx.x < SIMT_TILE) {
        int row = row0 + threadIdx.x;
        nb = row < n_out ? __ldg(a.nbr + (size_t)k * a.cap_out + row) : -1;
        sN[threadIdx.x] = nb;
      }
      if (!__syncthreads_or(nb >= 0)) continue;
      for (int e = threadIdx.x; e < SIMT_TILE * a.cin; e += 128) {
        int r = e / a.cin, ci = e - r * a.cin;
        int src = sN[r];
        sA[r][ci] = src >= 0 ? ld_as_float<TIN>(in + (size_t)src * a.cin + ci) : 0.f;
      }
      __syncthreads();
      const float* wk = a.w + (size_t)k * a.cin * COUT + co;
      for (int ci = 0; ci < a.cin; ++ci) {
        float w = __ldg(wk + (size_t)ci * COUT);
#pragma unroll
        for (int r = 0; r < RPT; ++r) acc[r] = fmaf(sA[rg * RPT + r][ci], w, acc[r]);
      }
      __syncthreads();
    }
    const float b = a.bias ? __ldg(a.bias + co) : 0.f;
#pragma unroll
    for (int r = 0; r < RPT; ++r) {
      int row = row0 + rg * RPT + r;
      if (row >= n_out) continue;
      float v = acc[r] + b;
      if (a.residual) v += ld_enc(a.residual, a.out_enc, (size_t)row, COUT, co);
      if (a.relu) v = fmaxf(v, 0.f);
      if (a.dense) {
        int4 q = __ldg(a.out_coors + row);
        size_t hw = (size_t)a.H * a.W;
        a.dense[((size_t)q.x * COUT * a.D + (size_t)co * a.D + q.y) * hw + (size_t)q.z * a.W + q.w] = v;
      } else {
        st_enc(a.out, a.out_enc, (size_t)row, COUT, co, v);
      }
    }
  }
}

// First layer of the encoder (conv_input: Cin = 4/5 raw voxel features -> 16): far too few
// input channels for a tensor-core tile.  One thread per output row keeps the COUT
// accumulators in registers, the whole (kvol, cin, COUT) weight set lives in shared memory
// and is read as broadcast float4; offsets without a neighbour are skipped per lane.
template <int COUT>
__global__ void __launch_bounds__(128) spconv_smallcin_kernel(ConvDev a) {
  extern __shared__ __align__(16) float sW[];   // kvol * cin * COUT
  const int nw = a.kvol * a.cin * COUT;
  for (int e = threadIdx.x; e < nw; e += blockDim.x) sW[e] = a.w[e];
  __syncthreads();
  const int n_out = a.d_n_out ? min(*a.d_n_out, a.cap_out) : a.cap_out;
  const float* in = (const float*)a.in;
  for (int row = blockIdx.x * blockDim.x + threadIdx.x; row < n_out; row += gridDim.x * blockDim.x) {
    float acc[COUT];
#pragma unroll
    for (int c = 0; c < COUT; ++c) acc[c] = a.bias ? __ldg(a.bias + c) : 0.f;
    // Offsets in batches of KB: the neighbour indices of the NEXT batch are requested before this batch's input rows, and the
    // (up to 8) input channels of the KB rows are independent predicated loads, so a row's latency chain is kvol / KB round
    // trips instead of 2 * kvol (the per-offset  index -> row -> FMA  loop measured 62 us for 160 k rows; accumulation order
    // unchanged: k ascending, ci ascending).
    constexpr int KB = 3, CMAX = 8;
    int nxt[KB];
#pragma unroll
    for (int j = 0; j < KB; ++j) nxt[j] = j < a.kvol ? __ldg(a.nbr + (size_t)j * a.cap_out + row) : -1;
    for (int k0 = 0; k0 < a.kvol; k0 += KB) {
      int src[KB];
#pragma unroll
      for (int j = 0; j < KB; ++j) {
        src[j] = nxt[j];
        nxt[j] = k0 + KB + j < a.kvol ? __ldg(a.nbr + (size_t)(k0 + KB + j) * a.cap_out + row) : -1;
      }
      float xv[KB][CMAX];
#pragma unroll
      for (int j = 0; j < KB; ++j) {
        const float* x = in + (size_t)max(src[j], 0) * a.cin;
#pragma unroll
        for (int ci = 0; ci < CMAX; ++ci) xv[j][ci] = (src[j] >= 0 && ci < a.cin) ? __ldg(x + ci) : 0.f;
      }
#pragma unroll
      for (int j = 0; j < KB; ++j) {
        if (src[j] < 0) continue;
        const float4* wk = reinterpret_cast<const float4*>(sW + (size_t)(k0 + j) * a.cin * COUT);
#pragma unroll
        for (int ci = 0; ci < CMAX; ++ci) {
          if (ci < a.cin) {
#pragma unroll
            for (int q = 0; q < COUT / 4; ++q) {
              const float4 w = wk[ci * (COUT / 4) + q];
              acc[4 * q + 0] = fmaf(xv[j][ci], w.x, acc[4 * q + 0]);
              acc[4 * q + 1] = fmaf(xv[j][ci], w.y, acc[4 * q + 1]);
              acc[4 * q + 2] = fmaf(xv[j][ci], w.z, acc[4 * q + 2]);
              acc[4 * q + 3] = fmaf(xv[j][ci], w.w, acc[4 * q + 3]);
            }
          }
        }
      }
    }
    if (a.relu) {
#pragma unroll
      for (int c = 0; c < COUT; ++c) acc[c] = fmaxf(acc[c], 0.f);
    }
    if (a.out_enc == SRF_F32) {
      float4* op = reinterpret_cast<float4*>((float*)a.out + (size_t)row * COUT);
#pragma unroll
      for (int c = 0; c < COUT; c += 4) op[c / 4] = make_float4(acc[c], acc[c + 1], acc[c + 2], acc[c + 3]);
    } else {
      const bool f16 = enc_is_f16(a.out_enc), split = enc_is_split(a.out_enc);
      uint16_t* orow = (uint16_t*)a.out + (size_t)row * COUT * (split ? 2 : 1);
#pragma unroll
      for (int c = 0; c < COUT; c += 8) {
        uint32_t h[4], l[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) split16x2(f16, acc[c + 2 * q], acc[c + 2 * q + 1], h[q], l[q]);
        *reinterpret_cast<uint4*>(orow + c) = make_uint4(h[0], h[1], h[2], h[3]);
        if (split) *reinterpret_cast<uint4*>(orow + COUT + c) = make_uint4(l[0], l[1], l[2], l[3]);
      }
    }
  }
}

// (kvol, cin, cout) f32 -> 16-bit elements in UMMA "core matrix" order, per kernel offset k and
// K chunk q of kc input channels:   [k][q][part][kc/8][co][ci%8]   (one 16-byte K-chunk per output
// channel row; part = hi only, or hi then lo for the split encodings); more than 128 output channels are
// laid out as column tiles [nt][k][q][part][kc/8][128][8]
__global__ void pack_weight_kernel(const float* __restrict__ w, int kvol, int cin, int cout, int kc, int tn, int enc,
                                   uint16_t* __restrict__ out) {
  const bool f16 = enc_is_f16(enc);
  const int parts = enc_is_split(enc) ? 2 : 1;
  int64_t total = (int64_t)kvol * cin * cout;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    int co = (int)(e % cout);
    int64_t t = e / cout;
    int ci = (int)(t % cin);
    int k = (int)(t / cin);
    const int q = ci / kc, cl = ci % kc;
    const int nt = co / tn, col = co % tn;                                   // column tiles of tn output channels
    const int64_t member = (((int64_t)nt * kvol + k) * (cin / kc) + q) * parts;   // in units of kc*tn elements
    const int64_t inner = ((int64_t)(cl / 8) * tn + col) * 8 + (cl % 8);
    const float v = w[e];
    const uint16_t h = pack16(f16, v);
    out[member * kc * tn + inner] = h;
    if (parts == 2) out[(member + 1) * kc * tn + inner] = pack16(f16, v - unpack16(f16, h));
  }
}

// nn.Linear weight (n, k) f32 -> 16-bit tiles [n/tn][k/tk][part][tk/8][tn][8]
__global__ void pack_linear_kernel(const float* __restrict__ w, int n, int k, int tn, int tk, int enc,
                                   uint16_t* __restrict__ out) {
  const bool f16 = enc_is_f16(enc);
  const int parts = enc_is_split(enc) ? 2 : 1;
  int64_t total = (int64_t)n * k;
  int nkc = k / tk;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    int kk = (int)(e % k);
    int nn = (int)(e / k);
    int nt = nn / tn, nl = nn % tn, kc = kk / tk, ci = kk % tk;
    const int64_t member = ((int64_t)nt * nkc + kc) * parts;
    const int64_t inner = ((int64_t)(ci / 8) * tn + nl) * 8 + (ci % 8);
    const float v = w[e];
    const uint16_t h = pack16(f16, v);
    out[member * tk * tn + inner] = h;
    if (parts == 2) out[(member + 1) * tk * tn + inner] = pack16(f16, v - unpack16(f16, h));
  }
}

// (rows, c) f32 -> rows of c_pad 16-bit elements (zero padded), split rows [hi(c_pad) | lo(c_pad)]
__global__ void convert_rows_kernel(const float* __restrict__ in, int64_t rows, int c, int c_pad, int enc,
                                    uint16_t* __restrict__ out) {
  const bool f16 = enc_is_f16(enc), split = enc_is_split(enc);
  int64_t total = rows * c_pad;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    int j = (int)(e % c_pad);
    int64_t r = e / c_pad;
    const float v = j < c ? in[r * c + j] : 0.f;
    const uint16_t h = pack16(f16, v);
    if (!split) { out[e] = h; continue; }
    out[r * 2 * c_pad + j] = h;
    out[r * 2 * c_pad + c_pad + j] = pack16(f16, v - unpack16(f16, h));
  }
}

// out[r] = in[perm[r]] for r < *d_n (rows of c floats): puts caller-ordered voxel features
// into the index's sorted row order (perm from srf_index_perm).
__global__ void gather_rows_kernel(const float* __restrict__ in, const int32_t* __restrict__ perm,
                                   const int32_t* __restrict__ d_n, int cap, int c, float* __restrict__ out) {
  int n = d_n ? min(*d_n, cap) : cap;
  int64_t total = (int64_t)n * c;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    int j = (int)(e % c);
    int64_t r = e / c;
    out[e] = __ldg(in + (size_t)__ldg(perm + r) * c + j);
  }
}

// ---- generic fp32 linear: out = epi(A (m,k) . W(n,k)^T + bias) ----------------------------
// block = 256 threads = 256 output columns (grid.y tiles n), LIN_ROWS rows (grid.x tiles m);
// A is staged through shared memory in K-chunks, each thread keeps LIN_ROWS accumulators.
constexpr int LIN_ROWS = 16;
constexpr int LIN_KC = 256;
__global__ void __launch_bounds__(256) linear_f32_kernel(const float* __restrict__ A, int m, int k,
                                                        const float* __restrict__ W, int n,
                                                        const float* __restrict__ bias, int relu,
                                                        float* __restrict__ out) {
  __shared__ float sa[LIN_ROWS][LIN_KC + 1];
  const int row0 = blockIdx.x * LIN_ROWS;
  const int col = blockIdx.y * 256 + threadIdx.x;
  float acc[LIN_ROWS];
#pragma unroll
  for (int r = 0; r < LIN_ROWS; ++r) acc[r] = 0.f;
  const float* wr = W + (size_t)(col < n ? col : 0) * k;
  for (int k0 = 0; k0 < k; k0 += LIN_KC) {
    const int kc = min(LIN_KC, k - k0);
    __syncthreads();
    for (int e = threadIdx.x; e < LIN_ROWS * LIN_KC; e += 256) {
      int r = e / LIN_KC, j = e - r * LIN_KC;
      sa[r][j] = (row0 + r < m && j < kc) ? A[(size_t)(row0 + r) * k + k0 + j] : 0.f;
    }
    __syncthreads();
    if (col < n) {
      for (int j = 0; j < kc; ++j) {
        float w = __ldg(wr + k0 + j);
#pragma unroll
        for (int r = 0; r < LIN_ROWS; ++r) acc[r] = fmaf(sa[r][j], w, acc[r]);
      }
    }
  }
  if (col >= n) return;
  const float b = bias ? bias[col] : 0.f;
#pragma unroll
  for (int r = 0; r < LIN_ROWS; ++r) {
    if (row0 + r >= m) continue;
    float v = acc[r] + b;
    if (relu) v = fmaxf(v, 0.f);
    out[(size_t)(row0 + r) * n + col] = v;
  }
}

// narrow outputs (n <= 16: class logits, box deltas): block = 16 rows x 16 columns, W transposed in shared memory
constexpr int SN_ROWS = 16, SN_MAXK = 512;
__global__ void __launch_bounds__(256) linear_smalln_kernel(const float* __restrict__ A, int m, int k, const float* __restrict__ W, int n,
                                                           const float* __restrict__ bias, int relu, float* __restrict__ out) {
  extern __shared__ float swt[];                       // [k][17]
  for (int e = threadIdx.x; e < n * k; e += blockDim.x) swt[(e % k) * 17 + e / k] = W[e];
  __syncthreads();
  const int col = threadIdx.x & 15, row = blockIdx.x * SN_ROWS + (threadIdx.x >> 4);
  if (row >= m || col >= n) return;
  const float* a = A + (size_t)row * k;
  float acc = 0.f;
  for (int j = 0; j < k; j += 4) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(a + j));
    acc = fmaf(v.x, swt[j * 17 + col], acc);
    acc = fmaf(v.y, swt[(j + 1) * 17 + col], acc);
    acc = fmaf(v.z, swt[(j + 2) * 17 + col], acc);
    acc = fmaf(v.w, swt[(j + 3) * 17 + col], acc);
  }
  acc += bias ? bias[col] : 0.f;
  out[(size_t)row * n + col] = relu ? fmaxf(acc, 0.f) : acc;
}

// row-wise LayerNorm (+ReLU) of (sum of split-K slabs + bias), one warp per row; f32 or bf16.
// The row is read once into registers (n <= 32*LN_MAXPL), then reduced with shuffles.
constexpr int LN_MAXPL = 16;   // values per lane -> n <= 512
template <int NPL>             // values per lane of this instantiation (n <= 32 * NPL): short rows get a short kernel
__global__ void layernorm_rows_kernel(const void* __restrict__ in, int in_enc, int64_t rows, int n, int n_partials,
                                      const float* __restrict__ bias, const float* __restrict__ resid, const float* __restrict__ g,
                                      const float* __restrict__ b, float eps, int relu, void* __restrict__ out, int out_enc,
                                      void* __restrict__ out2, int out2_enc) {
  int lane = threadIdx.x & 31;
  int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  float v[NPL];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NPL; ++i) {
    const int j = lane + 32 * i;
    v[i] = 0.f;
    if (j < n) {
      float t = ld_enc(in, in_enc, (size_t)row, n, j);
      for (int p = 1; p < n_partials; ++p) t += ld_enc(in, in_enc, (size_t)(p * rows + row), n, j);   // slab order: deterministic
      v[i] = t + (bias ? bias[j] : 0.f) + (resid ? resid[row * n + j] : 0.f);
      s += v[i];
    }
  }
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s / n;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NPL; ++i)
    if (lane + 32 * i < n) { float d = v[i] - mean; q += d * d; }
  for (int o = 16; o; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  const float rstd = rsqrtf(q / n + eps);
#pragma unroll
  for (int i = 0; i < NPL; ++i) {
    const int j = lane + 32 * i;
    if (j < n) {
      float y = (v[i] - mean) * rstd * g[j] + b[j];
      if (relu) y = fmaxf(y, 0.f);
      st_enc(out, out_enc, (size_t)row, n, j, y);
      if (out2) st_enc(out2, out2_enc, (size_t)row, n, j, y);
    }
  }
}

// One block per row, one thread per column (n <= 1024): used when split-K slabs have to be
// summed -- 4-32 warps per row instead of one keeps enough loads in flight.
__global__ void layernorm_cols_kernel(const void* __restrict__ in, int in_enc, int64_t rows, int n, int n_partials,
                                      const float* __restrict__ bias, const float* __restrict__ resid, const float* __restrict__ g,
                                      const float* __restrict__ b, float eps, int relu, void* __restrict__ out, int out_enc,
                                      void* __restrict__ out2, int out2_enc) {
  __shared__ float red[2][32];
  const int64_t row = blockIdx.x;
  const int j = threadIdx.x, lane = j & 31, w = j >> 5, nw = (blockDim.x + 31) >> 5;
  float v = 0.f;
  if (j < n) {
    for (int p = 0; p < n_partials; ++p) v += ld_enc(in, in_enc, (size_t)(p * rows + row), n, j);   // slab order: deterministic
    v += bias ? bias[j] : 0.f;
    v += resid ? resid[row * n + j] : 0.f;
  }
  float s = j < n ? v : 0.f;
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) red[0][w] = s;
  __syncthreads();
  float tot = 0.f;
  for (int i = 0; i < nw; ++i) tot += red[0][i];
  const float mean = tot / n;
  float d = j < n ? v - mean : 0.f;
  float q = d * d;
  for (int o = 16; o; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  if (lane == 0) red[1][w] = q;
  __syncthreads();
  float var = 0.f;
  for (int i = 0; i < nw; ++i) var += red[1][i];
  const float rstd = rsqrtf(var / n + eps);
  if (j < n) {
    float y = d * rstd * g[j] + b[j];
    if (relu) y = fmaxf(y, 0.f);
    st_enc(out, out_enc, (size_t)row, n, j, y);
    if (out2) st_enc(out2, out2_enc, (size_t)row, n, j, y);
  }
}

static int lgrid2(int64_t n, int threads) {
  int64_t g = (n + threads - 1) / threads;
  int64_t cap = (int64_t)sm_count() * 8;
  if (g > cap) g = cap;
  return g < 1 ? 1 : (int)g;
}

template <typename TIN>
static int launch_conv_f32(const ConvDev& d, int cout, int grid, cudaStream_t st) {
  switch (cout) {
    case 16: spconv_f32_kernel<16, TIN><<<grid, 128, 0, st>>>(d); break;
    case 32: spconv_f32_kernel<32, TIN><<<grid, 128, 0, st>>>(d); break;
    case 64: spconv_f32_kernel<64, TIN><<<grid, 128, 0, st>>>(d); break;
    case 128: spconv_f32_kernel<128, TIN><<<grid, 128, 0, st>>>(d); break;
    default: set_error("srf_spconv_f32: cout must be 16/32/64/128 (got %d)", cout); return SRF_ERR_UNSUPPORTED;
  }
  return SRF_OK;
}

}  // namespace srf

using namespace srf;

extern "C" {

int srf_spconv_f32(const srf_conv_args* a, void* stream) {
  SRF_CHECK_ARG(a && a->in && a->nbr && a->w && (a->out || a->dense), "srf_spconv_f32: null arg");
  // the kernels read rows of 4-byte (SRF_F32) or 2-byte bf16 (SRF_BF16) elements; any other encoding would be misread
  SRF_CHECK_ARG(a->in_dtype == SRF_F32 || a->in_dtype == SRF_BF16, "srf_spconv_f32: input features must be f32 or bf16 (got encoding %d)", a->in_dtype);
  SRF_CHECK_ARG(a->cin >= 1 && a->cin <= SIMT_MAXCIN, "srf_spconv_f32: cin must be in [1,%d]", SIMT_MAXCIN);
  SRF_CHECK_ARG(a->kvol >= 1 && a->kvol <= 27, "srf_spconv_f32: kvol must be in [1,27]");
  SRF_CHECK_ARG(a->cap_out > 0 && a->cap_out % 128 == 0, "srf_spconv_f32: cap_out must be a multiple of 128");
  SRF_CHECK_ARG(!a->dense || a->out_coors, "srf_spconv_f32: dense output needs out_coors");
  ConvDev d;
  d.in = a->in; d.nbr = a->nbr; d.tile_mask = a->tile_mask; d.d_n_out = a->d_n_out;
  d.w = (const float*)a->w; d.bias = a->bias; d.residual = a->residual; d.out = a->out; d.dense = a->dense;
  d.out_coors = (const int4*)a->out_coors; d.cin = a->cin; d.kvol = a->kvol; d.cap_out = a->cap_out;
  d.relu = a->relu; d.out_enc = a->dense ? SRF_F32 : a->out_dtype;
  d.D = a->out_dims[1]; d.H = a->out_dims[2]; d.W = a->out_dims[3];
  int ntiles = a->cap_out / SIMT_TILE;
  int grid = sm_count() * 8;
  if (grid > ntiles) grid = ntiles;
  cudaStream_t st = (cudaStream_t)stream;
  SRF_COUNT(1);
  if (a->in_dtype == SRF_F32 && a->cin <= 8 && (a->cout == 16 || a->cout == 32) && !a->residual && !a->dense) {
    // tiny-Cin first layer: thread-per-row kernel, weights in shared memory
    const size_t smem = (size_t)a->kvol * a->cin * a->cout * sizeof(float);
    int g2 = cdiv(a->cap_out, 128);
    if (g2 > sm_count() * 16) g2 = sm_count() * 16;
    if (a->cout == 16) spconv_smallcin_kernel<16><<<g2, 128, smem, st>>>(d);
    else spconv_smallcin_kernel<32><<<g2, 128, smem, st>>>(d);
    SRF_LAUNCH_CHECK();
    return SRF_OK;
  }
  int rc = a->in_dtype == SRF_BF16 ? launch_conv_f32<__nv_bfloat16>(d, a->cout, grid, st)
                                   : launch_conv_f32<float>(d, a->cout, grid, st);
  if (rc) return rc;
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

int srf_pack_weight_kc(int32_t cin, int32_t enc);   // igemm_umma.cu: K chunk per ring slot for (cin, enc)
int srf_conv_tile_n(int32_t cout);
int srf_linear_tile_k_enc(int32_t k, int32_t enc);
int srf_linear_tile_n(int32_t n);

int srf_pack_weight_tc(const float* w, int32_t kvol, int32_t cin, int32_t cout, int32_t enc, void* packed, void* stream) {
  SRF_CHECK_ARG(w && packed && kvol > 0 && cin % 8 == 0 && cout % 8 == 0 && enc_is_16(enc), "srf_pack_weight_tc: bad args");
  int64_t total = (int64_t)kvol * cin * cout;
  SRF_COUNT(1);
  pack_weight_kernel<<<lgrid2(total, 256), 256, 0, (cudaStream_t)stream>>>(w, kvol, cin, cout, srf_pack_weight_kc(cin, enc), srf_conv_tile_n(cout), enc, (uint16_t*)packed);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}
int srf_pack_weight_bf16(const float* w, int32_t kvol, int32_t cin, int32_t cout, void* packed, void* stream) {
  return srf_pack_weight_tc(w, kvol, cin, cout, SRF_BF16, packed, stream);
}

int srf_pack_linear_tc(const float* w, int32_t n, int32_t k, int32_t enc, void* packed, void* stream) {
  SRF_CHECK_ARG(w && packed && enc_is_16(enc), "srf_pack_linear_tc: bad args");
  int tk = srf_linear_tile_k_enc(k, enc), tn = srf_linear_tile_n(n);
  SRF_CHECK_ARG(k % tk == 0 && n % tn == 0 && tk % 16 == 0 && tn % 16 == 0,
                "srf_pack_linear_tc: n=%d k=%d not tileable (multiples of 16; of the tile size above it)", n, k);
  SRF_COUNT(1);
  pack_linear_kernel<<<lgrid2((int64_t)n * k, 256), 256, 0, (cudaStream_t)stream>>>(w, n, k, tn, tk, enc, (uint16_t*)packed);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}
int srf_pack_linear_bf16(const float* w, int32_t n, int32_t k, void* packed, void* stream) {
  return srf_pack_linear_tc(w, n, k, SRF_BF16, packed, stream);
}

int srf_convert_rows(const float* in, int64_t rows, int32_t c, int32_t c_pad, int32_t enc, void* out, void* stream) {
  SRF_CHECK_ARG(in && out && rows >= 0 && c > 0 && c_pad >= c && enc_is_16(enc), "srf_convert_rows: bad args");
  if (rows == 0) return SRF_OK;
  SRF_COUNT(1);
  convert_rows_kernel<<<lgrid2(rows * c_pad, 256), 256, 0, (cudaStream_t)stream>>>(in, rows, c, c_pad, enc, (uint16_t*)out);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}
int srf_f32_to_bf16(const float* in, int64_t rows, int32_t c, int32_t c_pad, void* out, void* stream) {
  return srf_convert_rows(in, rows, c, c_pad, SRF_BF16, out, stream);
}

int srf_gather_rows(const float* in, const int32_t* perm, const int32_t* d_n, int32_t cap, int32_t c, float* out,
                    void* stream) {
  SRF_CHECK_ARG(in && perm && out && cap >= 0 && c > 0, "srf_gather_rows: bad args");
  if (cap == 0) return SRF_OK;
  SRF_COUNT(1);
  gather_rows_kernel<<<lgrid2((int64_t)cap * c, 256), 256, 0, (cudaStream_t)stream>>>(in, perm, d_n, cap, c, out);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

int srf_linear_f32(const float* a, int32_t m, int32_t k, const float* w, int32_t n, const float* bias,
                   int32_t relu, float* out, void* stream) {
  SRF_CHECK_ARG(a && w && out && m >= 0 && k > 0 && n > 0, "srf_linear_f32: bad args");
  if (m == 0) return SRF_OK;
  SRF_COUNT(1);
  if (n <= 16 && k <= SN_MAXK && k % 4 == 0 && ((uintptr_t)a % 16 == 0)) {
    linear_smalln_kernel<<<cdiv(m, SN_ROWS), 256, (size_t)k * 17 * sizeof(float), (cudaStream_t)stream>>>(a, m, k, w, n, bias, relu, out);
    SRF_LAUNCH_CHECK();
    return SRF_OK;
  }
  dim3 grid(cdiv(m, LIN_ROWS), cdiv(n, 256));
  linear_f32_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(a, m, k, w, n, bias, relu, out);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

int srf_layernorm_enc(const void* in, int32_t in_enc, int64_t rows, int32_t n, int32_t n_partials, const float* bias,
                      const float* residual, const float* gamma, const float* beta, float eps, int32_t relu,
                      void* out, int32_t out_enc, void* out2, int32_t out2_enc, void* stream) {
  if (n_partials < 1) n_partials = 1;
  SRF_CHECK_ARG(in && out && gamma && beta && rows >= 0 && n > 0, "srf_layernorm: bad args");
  SRF_CHECK_ARG(in_enc == SRF_F32 || in_enc == SRF_BF16 || in_enc == SRF_F16, "srf_layernorm: input must be f32 / bf16 / f16");
  SRF_CHECK_ARG(n <= 32 * LN_MAXPL || (n_partials > 1 && n <= 1024), "srf_layernorm: n must be <= %d", 32 * LN_MAXPL);
  if (rows == 0) return SRF_OK;
  SRF_COUNT(1);
  if (n_partials > 1 && n <= 1024) {
    const int threads = (n + 31) / 32 * 32;
    layernorm_cols_kernel<<<(unsigned)rows, threads, 0, (cudaStream_t)stream>>>(in, in_enc, rows, n, n_partials, bias, residual, gamma, beta, eps, relu, out, out_enc, out2, out2_enc);
    SRF_LAUNCH_CHECK();
    return SRF_OK;
  }
  int wpb = 4;
  int grid = (int)((rows + wpb - 1) / wpb);
  if (n <= 128) layernorm_rows_kernel<4><<<grid, wpb * 32, 0, (cudaStream_t)stream>>>(in, in_enc, rows, n, n_partials, bias, residual, gamma, beta, eps, relu, out, out_enc, out2, out2_enc);
  else layernorm_rows_kernel<LN_MAXPL><<<grid, wpb * 32, 0, (cudaStream_t)stream>>>(in, in_enc, rows, n, n_partials, bias, residual, gamma, beta, eps, relu, out, out_enc, out2, out2_enc);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

int srf_layernorm(const void* in, int32_t dtype, int64_t rows, int32_t n, int32_t n_partials, const float* bias,
                  const float* gamma, const float* beta, float eps, int32_t relu, void* out, void* stream) {
  return srf_layernorm_enc(in, dtype, rows, n, n_partials, bias, nullptr, gamma, beta, eps, relu, out, dtype, nullptr, 0, stream);
}

}  // extern "C"
