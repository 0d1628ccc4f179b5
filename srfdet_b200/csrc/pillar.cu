// Pillar path of the srfdet_pillar_* configs (SURVEY.md 8f rank 4):
//   PillarFeatureNetCustom.forward (mmdet3d_plugin/models/voxel_encoders/pillar_encoder_custom.py:95-161)
//   with its single PFNLayer (voxel_encoders/utils.py:109-147; Linear(no bias) -> BN1d(eval) -> ReLU ->
//   max | avg over the T point slots) fused into one pass over the hard-voxelized pillars, and
//   mmdet3d PointPillarsScatter (cfg configs/nus/srfdet_pillar_nusc_L.py:53-54).
// srf_pillar_encode_rows joins the two with srf_nchw_to_rows for the detector: the PFN output of every pillar goes
// straight into its pixel row of the first SECONDCustom convolution's input, with no canvas in between.
// The decorated point features (raw C, offset to the pillar's point mean, offset to the pillar
// centre, optional range) never touch HBM; padded slots are zeroed AFTER decoration exactly like the
// reference (features *= mask), so a padded slot contributes relu(folded bias) to the max.
#include "common.cuh"

namespace srf {

constexpr int PILLAR_MAXT = 1024;   // point slots per pillar
constexpr int PILLAR_MAXF = 64;     // decorated features per point

struct PillarArgs {
  const float* voxels;      // (cap, T, C)
  const int32_t* num_points;
  const int32_t* coors;     // (cap, 4) b,z,y,x
  const int32_t* d_n;
  int cap, T, C;
  const float* w;           // (cout, F) Linear weight with BatchNorm folded
  const float* b;           // (cout) folded BatchNorm shift
  int cout, F;
  float vx, vy, vz, xo, yo, zo;
  int with_cluster, with_center, with_distance, legacy, avg;
  float* out;               // (cap, cout)
};

// ---- per-pillar math shared by srf_pillar_vfe and srf_pillar_encode_rows (same code, so the same bits) ----

// coordinate k of points_mean = features[:, :, :3].sum(dim=1) / num_points (padded slots are zeros, summed in slot order)
__device__ __forceinline__ float pillar_mean_coord(const float* pv, int T, int C, int k, int np) {
  float s = 0.f;
  for (int t = 0; t < T; ++t) s += __ldg(pv + t * C + k);
  return s / (float)np;
}

__device__ __forceinline__ float3 pillar_centre(const PillarArgs& a, const int32_t* cq) {
  return make_float3((float)__ldg(cq + 3) * a.vx + a.xo, (float)__ldg(cq + 2) * a.vy + a.yo, (float)__ldg(cq + 1) * a.vz + a.zo);
}

// The F decorated features of one point slot pt, in the Linear's input order, each passed to emit(value).  m is the
// slot's get_paddings_indicator mask: the decorated features of a padded slot are zeroed.
template <class Emit>
__device__ __forceinline__ void pillar_decorate(const PillarArgs& a, const float* pt, float m, float3 mean, float3 ctr, Emit&& emit) {
  const bool alias = a.with_center && a.legacy;
  const float x = __ldg(pt), y = __ldg(pt + 1), z = __ldg(pt + 2);
  const float cx = x - ctr.x, cy = y - ctr.y, cz = z - ctr.z;
  // legacy=True: f_center aliases features[:, :, :3] and is modified in place, so the raw xyz channels carry the
  // centre offsets too (pillar_encoder_custom.py:133-143)
  emit(m * (alias ? cx : x));
  emit(m * (alias ? cy : y));
  emit(m * (alias ? cz : z));
  for (int c = 3; c < a.C; ++c) emit(m * __ldg(pt + c));
  if (a.with_cluster) {
    emit(m * (x - mean.x));
    emit(m * (y - mean.y));
    emit(m * (z - mean.z));
  }
  if (a.with_center) {
    emit(m * cx);
    emit(m * cy);
    emit(m * cz);
  }
  if (a.with_distance) {
    const float dx = alias ? cx : x, dy = alias ? cy : y, dz = alias ? cz : z;
    emit(m * sqrtf(dx * dx + dy * dy + dz * dz));
  }
}

// One output channel of one pillar over the slots [t0, t1): red = max | sum of relu(w . dec_t + bias), the dot product
// accumulated with fmaf in feature order.  slot(t, emit) passes slot t's decorated features to emit; wt(j) is weight j
// of the channel.  Start from pillar_red_init, finish with pillar_red_out.
__device__ __forceinline__ float pillar_red_init(const PillarArgs& a) { return a.avg ? 0.f : -INFINITY; }

template <class Slot, class Wt>
__device__ __forceinline__ float pillar_reduce(const PillarArgs& a, float bias, int t0, int t1, float red, Slot&& slot, Wt&& wt) {
  for (int t = t0; t < t1; ++t) {
    int j = 0;
    float acc = 0.f;
    slot(t, [&](float v) { acc = fmaf(v, wt(j++), acc); });
    const float yv = fmaxf(acc + bias, 0.f);
    red = a.avg ? red + yv : fmaxf(red, yv);
  }
  return red;
}

__device__ __forceinline__ float pillar_red_out(const PillarArgs& a, float red, int np) { return a.avg ? red / (float)np : red; }

// one thread per (pillar, output channel): the T x F decorated features are recomputed by every channel's thread
// (a few hundred flops; the pillar's 100-odd input floats are L1 hits after the first thread) -- no staging, no
// dynamically indexed arrays.  Weights are read through the read-only cache (one row of F floats per thread).
__global__ void __launch_bounds__(256) pillar_vfe_kernel(const PillarArgs a) {
  const int n = a.d_n ? min(*a.d_n, a.cap) : a.cap;
  const long long total = (long long)n * a.cout;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(e / a.cout), co = (int)(e % a.cout);
    const float* pv = a.voxels + (size_t)v * a.T * a.C;
    const int np = __ldg(a.num_points + v);
    const float3 ctr = pillar_centre(a, a.coors + (size_t)v * 4);
    const float3 mean = make_float3(pillar_mean_coord(pv, a.T, a.C, 0, np), pillar_mean_coord(pv, a.T, a.C, 1, np),
                                    pillar_mean_coord(pv, a.T, a.C, 2, np));
    const float* wr = a.w + (size_t)co * a.F;
    const float red = pillar_reduce(
        a, __ldg(a.b + co), 0, a.T, pillar_red_init(a),
        [&](int t, auto&& emit) { pillar_decorate(a, pv + t * a.C, t < np ? 1.f : 0.f, mean, ctr, emit); },
        [&](int j) { return __ldg(wr + j); });
    a.out[e] = pillar_red_out(a, red, np);
  }
}

// srf_pillar_encode_rows: one warp per pillar.  Per chunk of 32 slots, lane t decorates slot t0 + t once into shared
// memory; then lane l reduces channels l, l + 32, ... over the chunk (partial reductions carried in shared memory between
// chunks), reading the weights transposed from shared memory.  Neighbouring lanes hold neighbouring channels, so even
// lanes store channel pairs through store_row_pair.
constexpr int ENC_WARPS = 4;
constexpr int ENC_MAX_COUT = 512;

struct PillarRowsArgs {
  PillarArgs p;             // p.voxels / num_points / coors: (n_blocks, cap, ...) blocks; p.d_n unused
  const int32_t* d_counts;  // (n_blocks)
  int n_blocks, ny, nx, enc;
  void* rows;
};

static inline __host__ __device__ int pillar_fp(int F) { return F | 1; }    // odd row pitch of the staged slots: conflict-free lane writes

static inline size_t pillar_rows_smem(int F, int cout) {
  return ((size_t)F * cout + (size_t)ENC_WARPS * (32 * pillar_fp(F) + cout)) * sizeof(float);
}

__global__ void __launch_bounds__(ENC_WARPS * 32) pillar_encode_rows_kernel(const PillarRowsArgs r) {
  extern __shared__ float sm[];
  const PillarArgs& a = r.p;
  const int FP = pillar_fp(a.F);
  float* s_w = sm;                                                 // (F, cout): w transposed
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* s_dec = s_w + (size_t)a.F * a.cout + (size_t)warp * (32 * FP + a.cout);   // (32, FP) decorated slots
  float* s_red = s_dec + 32 * FP;                                  // (cout) partial reductions of this warp's pillar
  for (int i = threadIdx.x; i < a.F * a.cout; i += blockDim.x) s_w[(i % a.F) * a.cout + i / a.F] = __ldg(a.w + i);
  __syncthreads();
  const int row_width = enc_is_split(r.enc) ? 2 * a.cout : a.cout;
  const int elem = r.enc == SRF_F32 ? 4 : 2;
  const long long total = (long long)r.n_blocks * a.cap;
  for (long long g = (long long)blockIdx.x * ENC_WARPS + warp; g < total; g += (long long)gridDim.x * ENC_WARPS) {
    const int b = (int)(g / a.cap), v = (int)(g % a.cap);
    if (v >= min(max(__ldg(r.d_counts + b), 0), a.cap)) continue;
    const size_t pil = (size_t)b * a.cap + v;
    const int4 q = __ldg(reinterpret_cast<const int4*>(a.coors) + pil);
    if (q.z < 0 || q.z >= r.ny || q.w < 0 || q.w >= r.nx) continue;   // off the grid: skipped like pillars_scatter_kernel
    const float* pv = a.voxels + pil * a.T * a.C;
    const int np = __ldg(a.num_points + pil);
    const float3 ctr = pillar_centre(a, a.coors + pil * 4);
    const float mk = lane < 3 ? pillar_mean_coord(pv, a.T, a.C, lane, np) : 0.f;
    const float3 mean = make_float3(__shfl_sync(0xffffffffu, mk, 0), __shfl_sync(0xffffffffu, mk, 1), __shfl_sync(0xffffffffu, mk, 2));
    char* row = static_cast<char*>(r.rows) + (((size_t)b * r.ny + q.z) * r.nx + q.w) * row_width * elem;
    for (int t0 = 0; t0 < a.T; t0 += 32) {
      const int t1 = min(t0 + 32, a.T), t = t0 + lane;
      if (t < t1) {
        float* d = s_dec + lane * FP;
        int j = 0;
        pillar_decorate(a, pv + t * a.C, t < np ? 1.f : 0.f, mean, ctr, [&](float x) { d[j++] = x; });
      }
      __syncwarp();
      for (int c0 = 0; c0 < a.cout; c0 += 32) {
        const int co = c0 + lane;
        float red = 0.f;
        if (co < a.cout) {
          red = pillar_reduce(
              a, __ldg(a.b + co), t0, t1, t0 == 0 ? pillar_red_init(a) : s_red[co],
              [&](int tt, auto&& emit) {
                const float* d = s_dec + (tt - t0) * FP;
                for (int j = 0; j < a.F; ++j) emit(d[j]);
              },
              [&](int j) { return s_w[j * a.cout + co]; });
          if (t1 < a.T) s_red[co] = red;
          else red = pillar_red_out(a, red, np);
        }
        if (t1 == a.T) {
          const float hi = __shfl_down_sync(0xffffffffu, red, 1);
          if (co < a.cout && (lane & 1) == 0) store_row_pair(r.enc, row, a.cout, co, red, hi);
        }
      }
      __syncwarp();
    }
  }
}

// PointPillarsScatter: canvas[b, c, y, x] = feats[row, c] (canvas zeroed by the caller).
// channels_last: the canvas is (B, ny, nx, C) in memory (a torch.channels_last tensor).
__global__ void pillars_scatter_kernel(const float* __restrict__ feats, const int32_t* __restrict__ coors, const int32_t* __restrict__ d_n,
                                       int cap, int c, int ny, int nx, int channels_last, float* __restrict__ canvas) {
  const int n = d_n ? min(*d_n, cap) : cap;
  const int64_t total = (int64_t)n * c;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int row = (int)(e / c), ch = (int)(e % c);
    const int4 q = __ldg(reinterpret_cast<const int4*>(coors) + row);
    if (q.x < 0 || q.z < 0 || q.z >= ny || q.w < 0 || q.w >= nx) continue;
    const size_t cell = (size_t)q.z * nx + q.w;
    const size_t dst = channels_last ? ((size_t)q.x * ny * nx + cell) * c + ch : ((size_t)q.x * c + ch) * ny * nx + cell;
    canvas[dst] = __ldg(feats + e);
  }
}

}  // namespace srf

using namespace srf;

extern "C" {

// PillarArgs of the two PFN entries; nonzero (error set) on an unsupported shape
static int pillar_args(const char* who, PillarArgs& a, const float* voxels, const int32_t* num_points, const int32_t* coors,
                       int32_t cap, int32_t t, int32_t c, const float* w_folded, const float* b_folded, int32_t cout,
                       const float voxel_size[3], const float offsets[3], int32_t flags) {
  SRF_CHECK_ARG(voxels && num_points && coors && w_folded && b_folded && voxel_size && offsets, "%s: null arg", who);
  SRF_CHECK_ARG(cap >= 0 && t >= 1 && t <= PILLAR_MAXT && c >= 3 && c <= 8 && cout >= 1,
                "%s: need 1 <= T <= %d, 3 <= C <= 8", who, PILLAR_MAXT);
  a = PillarArgs{};
  a.voxels = voxels; a.num_points = num_points; a.coors = coors; a.cap = cap; a.T = t; a.C = c;
  a.w = w_folded; a.b = b_folded; a.cout = cout;
  a.vx = voxel_size[0]; a.vy = voxel_size[1]; a.vz = voxel_size[2];
  a.xo = offsets[0]; a.yo = offsets[1]; a.zo = offsets[2];
  a.with_cluster = flags & 1; a.with_center = (flags >> 1) & 1; a.with_distance = (flags >> 2) & 1;
  a.legacy = (flags >> 3) & 1; a.avg = (flags >> 4) & 1;
  a.F = c + (a.with_cluster ? 3 : 0) + (a.with_center ? 3 : 0) + (a.with_distance ? 1 : 0);
  SRF_CHECK_ARG(a.F <= PILLAR_MAXF, "%s: too many decorated features", who);
  return SRF_OK;
}

int srf_pillar_vfe(const float* voxels, const int32_t* num_points, const int32_t* coors, int32_t cap, const int32_t* d_n,
                   int32_t t, int32_t c, const float* w_folded, const float* b_folded, int32_t cout, const float voxel_size[3],
                   const float offsets[3], int32_t flags, float* out, void* stream) {
  SRF_CHECK_ARG(out, "srf_pillar_vfe: null arg");
  PillarArgs a;
  const int rc = pillar_args("srf_pillar_vfe", a, voxels, num_points, coors, cap, t, c, w_folded, b_folded, cout, voxel_size,
                             offsets, flags);
  if (rc != SRF_OK) return rc;
  if (cap == 0) return SRF_OK;
  a.out = out;
  a.d_n = d_n;
  long long g = ((long long)cap * cout + 255) / 256;
  if (g > sm_count() * 16) g = sm_count() * 16;
  SRF_COUNT(1);
  pillar_vfe_kernel<<<(int)g, 256, 0, (cudaStream_t)stream>>>(a);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

int srf_pillar_encode_rows(const float* voxels, const int32_t* num_points, const int32_t* coors, const int32_t* d_counts,
                           int32_t n_blocks, int32_t block_rows, int32_t t, int32_t c, const float* w_folded,
                           const float* b_folded, int32_t cout, const float voxel_size[3], const float offsets[3], int32_t flags,
                           int32_t ny, int32_t nx, int32_t enc, void* rows, void* stream) {
  SRF_CHECK_ARG(d_counts && rows && n_blocks >= 1 && ny >= 1 && nx >= 1 && enc >= SRF_F32 && enc <= SRF_F16X2,
                "srf_pillar_encode_rows: bad args");
  SRF_CHECK_ARG(cout <= ENC_MAX_COUT, "srf_pillar_encode_rows: need cout <= %d", ENC_MAX_COUT);
  PillarRowsArgs r = {};
  const int rc = pillar_args("srf_pillar_encode_rows", r.p, voxels, num_points, coors, block_rows, t, c, w_folded, b_folded,
                             cout, voxel_size, offsets, flags);
  if (rc != SRF_OK) return rc;
  r.d_counts = d_counts; r.n_blocks = n_blocks; r.ny = ny; r.nx = nx; r.enc = enc; r.rows = rows;
  cudaStream_t st = (cudaStream_t)stream;
  SRF_CUDA(cudaMemsetAsync(rows, 0, (size_t)n_blocks * ny * nx * enc_row_bytes(enc, cout), st));
  if (block_rows == 0) return SRF_OK;
  const size_t smem = pillar_rows_smem(r.p.F, cout);
  if (smem > 48 * 1024) SRF_CUDA(cudaFuncSetAttribute(pillar_encode_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  long long g = ((long long)n_blocks * block_rows + ENC_WARPS - 1) / ENC_WARPS;
  if (g > sm_count() * 16) g = sm_count() * 16;
  SRF_COUNT(1);
  pillar_encode_rows_kernel<<<(int)g, ENC_WARPS * 32, smem, st>>>(r);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

int srf_pillars_scatter(const float* feats, const int32_t* coors, int32_t cap, const int32_t* d_n, int32_t c, int32_t ny,
                        int32_t nx, int32_t channels_last, float* canvas, void* stream) {
  SRF_CHECK_ARG(feats && coors && canvas && cap >= 0 && c >= 1 && ny >= 1 && nx >= 1, "srf_pillars_scatter: bad args");
  if (cap == 0) return SRF_OK;
  int64_t total = (int64_t)cap * c;
  int64_t g = (total + 255) / 256;
  if (g > sm_count() * 16) g = sm_count() * 16;
  SRF_COUNT(1);
  pillars_scatter_kernel<<<(int)g, 256, 0, (cudaStream_t)stream>>>(feats, coors, d_n, cap, c, ny, nx, channels_last, canvas);
  SRF_LAUNCH_CHECK();
  return SRF_OK;
}

}  // extern "C"
