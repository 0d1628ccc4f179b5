/*
 * srfdet_b200.h -- C ABI of libsrfdet_b200.so: the sm_100a kernels behind the
 * mmdet3d_plugin drop-in modules (srfdet_b200/plugin/*.py).
 *
 * The reference (gopi-erabati/SRFDet3D) has no FFI of its own: its boundary to native
 * code is the set of third-party Python ops it calls.  Each entry point below names the
 * reference call site (file:line under /root/reference) and the third-party op it
 * replaces.  INTEGRATION.md shows the ctypes binding a maintainer adds.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless the name ends in _host; buffers are
 *    caller-allocated (torch tensors); the library never allocates device memory.
 *  - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, no host
 *    synchronisation happens inside any call.
 *  - counts produced on the device stay on the device (int32_t* d_...); kernels that
 *    consume them are launched over a host-known capacity and read the count themselves,
 *    so a whole frame can be enqueued (or graph-captured) without a host round trip.
 *  - return 0 on success; otherwise a negative code and srf_last_error() (thread-local
 *    string).  No exceptions cross the boundary.
 *  - coordinates are int32 (b, z, y, x) as in mmcv / spconv.
 */
#ifndef SRFDET_B200_H_
#define SRFDET_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SRF_OK 0
#define SRF_ERR_ARG (-1)
#define SRF_ERR_CUDA (-2)
#define SRF_ERR_UNSUPPORTED (-3)

/* Element encodings of activation / weight buffers.
 *  SRF_F32, SRF_BF16, SRF_F16: plain rows of c elements.
 *  SRF_BF16X2 / SRF_F16X2 ("split"): a row of c values is stored as 2c 16-bit elements
 *  [hi(c) | lo(c)] with value = hi + lo (hi = round16(v), lo = round16(v - hi)).  The tensor-core
 *  kernels multiply split operands with three MMAs (Ah.Wh + Al.Wh + Ah.Wl, fp32 accumulate),
 *  which reproduces fp32 products to ~2^-16 (bf16) / 2^-21 (f16) relative: the tensor-core form
 *  of the reference's FP32 mode (srfdet.py:204-206 force_fp32).  SRF_F16 is the reference's own
 *  half precision (sparse_encoder_custom.py:109 auto_fp16); stores saturate at +-65504. */
#define SRF_F32 0
#define SRF_BF16 1
#define SRF_F16 2
#define SRF_BF16X2 3
#define SRF_F16X2 4

int srf_version(void);
const char* srf_last_error(void);
/* number of SMs of the current device (grid sizing of the persistent kernels) */
int srf_sm_count(void);
/* kernels launched by this library since load (host counter; bench.py's gpu_launches) */
unsigned long long srf_launch_count(void);

/* ---------------------------------------------------------------------------------- *
 * Voxel geometry.  Replaces mmcv/ops/voxelize.py grid computation
 * (call site: mmdet3d_plugin/models/detectors/srfdet.py:58).
 * ---------------------------------------------------------------------------------- */
typedef struct srf_geom {
  float vs[3];     /* voxel size x,y,z */
  float lo[3];     /* range min x,y,z */
  float hi[3];     /* range max x,y,z */
  int32_t grid[3]; /* cells x,y,z = round((hi-lo)/vs) in fp32 */
} srf_geom;
int srf_geom_init(srf_geom* g_host, const float voxel_size_host[3], const float pc_range_host[6]);

/* Dynamic voxelization: replaces mmcv dynamic_voxelize_forward
 * (srfdet.py:238; batch-index padding of srfdet.py:242-246 fused when batch_idx >= 0).
 * coors: (n,3) (z,y,x) when batch_idx < 0, else (n,4) (b,z,y,x); invalid points -> -1s. */
int srf_dynamic_voxelize(const float* points, int32_t n, int32_t c, const srf_geom* g_host,
                         int32_t batch_idx, int32_t* coors, void* stream);

/* Hard voxelization: replaces mmcv hard_voxelize_forward (deterministic) (srfdet.py:221)
 * and, when `mean` is given, HardSimpleVFE (cfg configs/nus/srfdet_voxel_nusc_L.py:40).
 *  voxels      (max_voxels, max_points, c) f32, zero padded   [nullable]
 *  coors       (max_voxels, 3) zyx, or (max_voxels, 4) bzyx when batch_idx >= 0
 *  num_points  (max_voxels)
 *  mean        (max_voxels, c) f32 = sum of kept points / num_points       [nullable]
 *  point2voxel (n) voxel id that stored the point, -1 if dropped          [nullable]
 *  d_voxel_num device scalar: number of voxels produced (<= max_voxels)
 * Rows >= *d_voxel_num of the outputs are left untouched. */
size_t srf_hard_voxelize_ws_bytes(int32_t n, int32_t max_points, int32_t max_voxels);
int srf_hard_voxelize(const float* points, int32_t n, int32_t c, const srf_geom* g_host,
                      int32_t max_points, int32_t max_voxels, int32_t batch_idx, float* voxels,
                      int32_t* coors, int32_t* num_points, float* mean, int32_t* point2voxel,
                      int32_t* d_voxel_num, void* ws, size_t ws_bytes, void* stream);

/* Hard voxelization of B clouds in one launch sequence (the number of launches does not depend
 * on B).  Cloud b is points_host[b] (n_host[b], c) on the device; host arrays of B entries.
 * Block b of every output equals, bit for bit, what srf_hard_voxelize(..., batch_idx = b)
 * writes for cloud b alone (its first-come voxel order, slots, counts, coordinates and means):
 *  voxels      (B, max_voxels, max_points, c) f32, zero padded   [nullable]
 *  coors       (B, max_voxels, 4) bzyx, b = block index
 *  num_points  (B, max_voxels)
 *  mean        (B, max_voxels, c) f32                            [nullable]
 *  d_counts    (B) device: voxels of each block (<= max_voxels)
 * Rows of block b at and past d_counts[b] are left untouched.  Limits (SRF_ERR_ARG, before any
 * launch): 1 <= B <= SRF_HV_BATCH_MAX, 3 <= c <= 8, the row counts sum to < 2^31, and
 * B x max_voxels and B x table capacity (the power of two >= max(1024, 2 max n)) < 2^31.
 * Workspace: srf_hard_voxelize_batch_ws_bytes(n_host, B, ...) bytes, 0 for bad arguments; one
 * hash table per cloud, so it is about B times the largest cloud's srf_hard_voxelize workspace
 * (B = 32 clouds of 300k points, max_points 10, 160k voxels: 723 MB).  No allocation, no host
 * synchronisation: a captured call replays.  11 launches (10 without voxels), 2 of them memsets. */
#define SRF_HV_BATCH_MAX 1024
size_t srf_hard_voxelize_batch_ws_bytes(const int32_t* n_host, int32_t batch, int32_t max_points, int32_t max_voxels);
int srf_hard_voxelize_batch(const float* const* points_host, const int32_t* n_host, int32_t batch, int32_t c,
                            const srf_geom* g_host, int32_t max_points, int32_t max_voxels, float* voxels,
                            int32_t* coors, int32_t* num_points, float* mean, int32_t* d_counts, void* ws,
                            size_t ws_bytes, void* stream);

/* Batched hard voxelization without a host read of the per-sample voxel counts: the
 * reference voxelizes each sample alone and concatenates the valid rows (srfdet.py:218-232);
 * here every sample writes a fixed block of block_rows rows (srf_hard_voxelize with its own
 * d_voxel_num) and this call packs the valid rows of all blocks, in block order, in one launch.
 * For each of the n_arrays arrays (4-byte elements): row r < min(d_counts[b], block_rows) of
 * block b is row (b * block_rows + r) of `src` (rows src_ld elements apart); its first `width`
 * elements go to row (sum_{j<b} min(d_counts[j], block_rows) + r) of `dst` (rows dst_ld apart).
 * d_total (device scalar) = number of packed rows.  Output rows >= *d_total are left untouched:
 * consumers read the count (e.g. the sparse encoder's d_n).  src and dst must not overlap.
 * No allocation, no host synchronisation (capturable in a CUDA graph). */
#define SRF_CONCAT_MAX_ARRAYS 4
typedef struct srf_rows {
  const void* src;
  void* dst;
  int32_t src_ld;
  int32_t dst_ld;
  int32_t width;
} srf_rows;
int srf_concat_counted_rows(const int32_t* d_counts, int32_t n_blocks, int32_t block_rows,
                            const srf_rows* arrays_host, int32_t n_arrays, int32_t* d_total, void* stream);

/* ---------------------------------------------------------------------------------- *
 * Cell index: occupancy bitmap + per-word rank over a dense (B,Z,Y,X) grid.  rank(cell)
 * enumerates occupied cells in ascending linear order, i.e. lexicographic (b,z,y,x):
 * exactly the order of at::unique_dim in mmcv DynamicScatter and the canonical rulebook
 * order (SURVEY.md 8a).  It replaces: the sort in DynamicPointToVoxelForward, the dense
 * canvas of map_voxel_center_to_point (voxel_encoder.py:118-158) and spconv's hash table.
 * ---------------------------------------------------------------------------------- */
size_t srf_index_bytes(int64_t ncells);
int srf_index_clear(void* index, int64_t ncells, void* stream);
/* set the bit of every row of coors (n,4); rows with a negative entry are skipped.
 * d_n (nullable) overrides n with a device-side count (n is then the capacity). */
int srf_index_mark(void* index, const int32_t dims_host[4], const int32_t* coors, int32_t n,
                   const int32_t* d_n, void* stream);
/* mark the outputs of a strided sparse conv: o = (p + pad - k)/stride where divisible
 * (spconv pair rule; sparse_encoder_custom.py:99-107,172-194).  dims are the OUTPUT dims. */
int srf_index_mark_strided(void* out_index, const int32_t out_dims_host[4], const int32_t* in_coors,
                           int32_t cap_in, const int32_t* d_n_in, const int32_t ksize_host[3],
                           const int32_t stride_host[3], const int32_t pad_host[3], void* stream);
/* popcount scan -> ranks; *d_num = number of occupied cells */
int srf_index_finalize(void* index, int64_t ncells, int32_t* d_num, void* stream);
/* coors_out (cap,4): coordinates of the occupied cells in rank order */
int srf_index_emit_coors(const void* index, const int32_t dims_host[4], int32_t* coors_out,
                         int32_t cap, void* stream);
/* rows[i] = rank of coors[i] or -1 (absent / negative coordinate) */
int srf_index_lookup(const void* index, const int32_t dims_host[4], const int32_t* coors, int32_t n,
                     const int32_t* d_n, int32_t* rows, void* stream);
/* perm[rank(coors[i])] = i  (rank -> caller's row order) */
int srf_index_perm(const void* index, const int32_t dims_host[4], const int32_t* coors, int32_t n,
                   const int32_t* d_n, int32_t* perm, void* stream);

/* out[r,:] = in[perm[r],:] for r < *d_n (cap rows when d_n is null); rows of c floats.
 * Brings caller-ordered voxel features (SparseEncoderCustom.forward input,
 * sparse_encoder_custom.py:110-124) into the index's sorted row order. */
int srf_gather_rows(const float* in, const int32_t* perm, const int32_t* d_n, int32_t cap, int32_t c,
                    float* out, void* stream);

/* ---------------------------------------------------------------------------------- *
 * DynamicScatter: replaces mmcv dynamic_point_to_voxel_forward
 * (voxel_encoder.py:82,99-102,189,232).  mode 0 = max, 1 = mean.  coor_dim 3 or 4.
 * dims_host = (B,Z,Y,X) of the voxel grid (B = 1 for coor_dim 3).
 * Outputs have capacity n rows; *d_num_voxels rows are valid, sorted like unique_dim.
 * point2voxel (n) [nullable].  ws: srf_scatter_ws_bytes.
 * ---------------------------------------------------------------------------------- */
size_t srf_scatter_ws_bytes(int64_t ncells, int32_t n, int32_t c);
int srf_dynamic_scatter(const float* feats, const int32_t* coors, int32_t n, int32_t c,
                        int32_t coor_dim, const int32_t dims_host[4], int32_t mode,
                        float* out_feats, int32_t* out_coors, int32_t* d_num_voxels,
                        int32_t* point2voxel, void* ws, size_t ws_bytes, void* stream);

/* DynamicVFECustom.forward, eval mode, fused (voxel_encoder.py:162-240 with
 * map_voxel_center_to_point :118-158, DynamicVFELayer utils.py:8-45 and the eval path of
 * NaiveSyncBatchNorm1dCustom ops/norm.py:57-58 folded into the weights).
 *  points (n,cin), coors (n,4)    pos_w0 (32,3) pos_b0 (32) pos_w1 (32,32) pos_b1 (32)
 *  vfe_w0 (c0, cin+35) vfe_b0 (c0); vfe_w1 (c1, 2*c0) vfe_b1 (c1) [nullable: one layer]
 *  out_feats (n, c_last), out_coors (n,4): *d_num_voxels valid rows. */
typedef struct srf_vfe_params {
  const float *pos_w0, *pos_b0, *pos_w1, *pos_b1;
  const float *vfe_w0, *vfe_b0, *vfe_w1, *vfe_b1;
  int32_t cin, c0, c1; /* c1 = 0 when there is a single VFE layer */
  float vx, vy, vz, x_off, y_off, z_off;
} srf_vfe_params;
size_t srf_dynamic_vfe_ws_bytes(int64_t ncells, int32_t n);
int srf_dynamic_vfe(const float* points, const int32_t* coors, int32_t n, const int32_t dims_host[4],
                    const srf_vfe_params* p_host, float* out_feats, int32_t* out_coors,
                    int32_t* d_num_voxels, void* ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------------- *
 * Pillar path (srfdet_pillar_* configs).
 * srf_pillar_vfe: PillarFeatureNetCustom.forward with its single PFNLayer fused
 *   (voxel_encoders/pillar_encoder_custom.py:95-161, voxel_encoders/utils.py:109-147):
 *   voxels (cap, t, c) zero-padded pillars from srf_hard_voxelize, num_points (cap), coors (cap,4)
 *   (b,z,y,x); decoration (cluster offset, pillar-centre offset, range) -> mask -> Linear (BatchNorm1d
 *   folded: w_folded (cout, F), b_folded (cout)) -> ReLU -> max | mean over the t slots -> out (cap, cout).
 *   flags: bit0 with_cluster_center, bit1 with_voxel_center, bit2 with_distance, bit3 legacy, bit4 avg.
 *   offsets = (vx/2 + x_min, vy/2 + y_min, vz/2 + z_min).  d_n (nullable): device row count.
 * srf_pillars_scatter: mmdet3d PointPillarsScatter (cfg configs/nus/srfdet_pillar_nusc_L.py:53-54):
 *   canvas (B, c, ny, nx) f32 (zeroed by the caller; (B, ny, nx, c) in memory when channels_last).
 * ---------------------------------------------------------------------------------- */
int srf_pillar_vfe(const float* voxels, const int32_t* num_points, const int32_t* coors, int32_t cap,
                   const int32_t* d_n, int32_t t, int32_t c, const float* w_folded, const float* b_folded,
                   int32_t cout, const float voxel_size_host[3], const float offsets_host[3], int32_t flags,
                   float* out, void* stream);
int srf_pillars_scatter(const float* feats, const int32_t* coors, int32_t cap, const int32_t* d_n, int32_t c,
                        int32_t ny, int32_t nx, int32_t channels_last, float* canvas, void* stream);
/* srf_pillar_encode_rows: srf_pillar_vfe -> srf_pillars_scatter -> srf_nchw_to_rows in one pass, bit for bit, for a
 *   batch of n_blocks per-sample blocks as srf_hard_voxelize writes them: voxels (n_blocks, block_rows, t, c),
 *   num_points (n_blocks, block_rows), coors (n_blocks, block_rows, 4) (b,z,y,x), d_counts (n_blocks) device counts.
 *   Pillars are the rows v < clamp(d_counts[b], 0, block_rows) of block b; the batch index is the block index (the
 *   b column of coors is not read); pillars whose (y, x) is off the ny x nx grid are skipped.
 *   rows (>= n_blocks*ny*nx rows of enc_width(enc, cout) elements, enc any of SRF_F32 .. SRF_F16X2): row
 *   (b*ny + y)*nx + x holds the PFN output of block b's pillar at (y, x), encoded like srf_nchw_to_rows (SRF_F32:
 *   plain); every other row below n_blocks*ny*nx is zero.  Rows from n_blocks*ny*nx on (e.g. the 128-row padding of
 *   the backbone's row buffers) are left untouched.  Same flags / weights / limits as srf_pillar_vfe, and cout <= 512.
 *   Two launches (zero, write), no allocation, no host synchronisation (capturable in a CUDA graph). */
int srf_pillar_encode_rows(const float* voxels, const int32_t* num_points, const int32_t* coors, const int32_t* d_counts,
                           int32_t n_blocks, int32_t block_rows, int32_t t, int32_t c, const float* w_folded,
                           const float* b_folded, int32_t cout, const float voxel_size_host[3], const float offsets_host[3],
                           int32_t flags, int32_t ny, int32_t nx, int32_t enc, void* rows, void* stream);

/* ---------------------------------------------------------------------------------- *
 * Rulebook: replaces spconv get_indice_pairs for SubMConv3d / SparseConv3d
 * (sparse_encoder_custom.py:84-107,165-215).  Output-stationary form:
 *   nbr[k * cap_out + o] = input row feeding output row o through kernel offset k
 *   (k = (kz*KH + ky)*KW + kx, input cell = o*stride - pad + k), or -1.
 *   tile_mask[o / 128] bit k set iff some row of that 128-row tile has a neighbour at k.
 *   The conv kernels may skip offsets whose bit is clear, so a superset of this mask is also
 *   valid; a live tile with no bit set (no row has any neighbour) yields act(bias (+ residual)).
 * in_perm (nullable) maps input rank -> caller row (first layer, unsorted input rows).
 * ---------------------------------------------------------------------------------- */
int srf_rulebook_build(const void* in_index, const int32_t in_dims_host[4], const int32_t* in_perm,
                       const int32_t* out_coors, int32_t cap_out, const int32_t* d_n_out,
                       const int32_t ksize_host[3], const int32_t stride_host[3],
                       const int32_t pad_host[3], int32_t* nbr, uint32_t* tile_mask, void* stream);

/* Rulebook of a dense 2-D conv (ksize x ksize, stride, zero padding) over (n, h, w) pixel rows in
 * row-major order: lets the BEV backbone / neck convolutions (SECONDCustom, FPN;
 * models/backbones/second_custom.py:23-91) run on srf_spconv_tc over NHWC activations.
 * nbr (ksize*ksize, cap_out), cap_out a multiple of 128 >= n*ho*wo. */
int srf_dense_rulebook(int32_t n, int32_t h, int32_t w, int32_t ksize, int32_t stride, int32_t pad,
                       int32_t cap_out, int32_t* nbr, uint32_t* tile_mask, void* stream);

/* (n, c, h, w) f32 NCHW (the layout SparseConvTensor.dense() emits) -> (n*h*w, c) pixel rows in a 16-bit
 * encoding: the A operand of the first backbone convolution. */
int srf_nchw_to_rows(const float* in, int32_t n, int32_t c, int32_t h, int32_t w, int32_t enc, void* out,
                     void* stream);
/* FPN top-down step on pixel rows in encoding enc: rows_hi (n,h,w,c) += nearest_upsample(rows_lo (n,h_lo,w_lo,c))
 * (mmdet FPN.forward: F.interpolate(size=, mode='nearest')). */
int srf_upsample_add(void* rows_hi, const void* rows_lo, int32_t n, int32_t h, int32_t w, int32_t h_lo,
                     int32_t w_lo, int32_t c, int32_t enc, void* stream);

/* Dense 3x3 / stride 1 / pad 1 convolution + folded BatchNorm2d (+ReLU) over NHWC pixel rows: the stride-1 ConvModules of
 * SECONDCustom (mmdet3d_plugin/models/backbones/second_custom.py:23-91, cfg configs/nus/srfdet_voxel_nusc_L.py:55-66) and
 * the FPN output convs (:67-75).  in: (n*h*w, cin) rows in SRF_F16 / SRF_BF16, cin a multiple of 128 (<= 512); w_packed:
 * srf_pack_weight_tc(kvol = 9 in (ky, kx) order, cin, cout, enc) with BN folded; cout a multiple of 128; out (n*h*w, cout)
 * rows in out_enc (SRF_F32 or a 16-bit form of the input's element format).  The 18 x 10 input halo of a 16 x 8 pixel tile
 * is staged once in shared memory and the nine kernel offsets are nine tcgen05 descriptor offsets into it (csrc/conv3x3_halo.cu).
 * Returns SRF_ERR_UNSUPPORTED for any other shape / encoding: callers then use srf_spconv_tc over srf_dense_rulebook. */
int srf_conv3x3_rows(const void* in, int32_t enc, int32_t n, int32_t h, int32_t w, int32_t cin, const void* w_packed,
                     int32_t cout, const float* bias, int32_t relu, void* out, int32_t out_enc, void* stream);
/* 1 when the last srf_conv3x3_rows launch staged its halos with TMA tensor copies (cp.async.bulk.tensor.5d, out-of-image
 * pixels zero-filled by the copy engine), 0 when it used the cp.async gather producers (tensor-map encoder unavailable or
 * SRF_HALO_TMA=0), -1 before the first launch. */
int srf_conv3x3_last_used_tma(void);

/* ---------------------------------------------------------------------------------- *
 * Sparse convolution + folded BatchNorm1d + residual + ReLU (+ dense scatter).
 * Replaces spconv SubMConv3d/SparseConv3d forward, BN1d, ReLU, SparseBasicBlock residual
 * and SparseConvTensor.dense() (sparse_encoder_custom.py:125-138).
 *   out[o] = act( sum_k W_k^T in[nbr[k][o]] + bias (+ residual[o]) )
 * srf_spconv_f32: SIMT FFMA, fp32 (cross-check mode; also the few-channel first layer of every
 *            mode: in f32, out in any encoding).  in_dtype SRF_F32 or SRF_BF16 only (any other
 *            encoding returns SRF_ERR_ARG); cin in [1,128], cout in {16,32,64,128}; out_dtype and
 *            the residual's encoding: any of the five.  w (kvol, cin, cout) f32.
 * srf_spconv_tc : tcgen05/TMEM implicit GEMM, fp32 accumulate.  in_dtype SRF_BF16 | SRF_F16 (one MMA
 *            per product) or SRF_BF16X2 | SRF_F16X2 (hi + lo operands, three MMAs per product: the
 *            tensor-core form of the reference's FP32 mode).  out_dtype: the same encoding, or
 *            SRF_F32.  w packed by srf_pack_weight_tc for the same encoding.  cin in
 *            {16,32,64,128,256}, cout in {16,32,64,128} or a multiple of 128 (column tiles).  srf_spconv_bf16 / srf_pack_weight_bf16: the SRF_BF16 forms (round 1 names).
 * dense (nullable): write the result into a zeroed (B, cout*D, H, W) f32 map instead of
 * `out` (needs out_coors + out_dims_host).
 * ---------------------------------------------------------------------------------- */
typedef struct srf_conv_args {
  const void* in;          /* (in_rows, cin) in in_dtype (split encodings: 2*cin 16-bit elements per row) */
  int32_t in_dtype;        /* SRF_* encoding */
  int32_t in_rows;         /* rows allocated behind `in` (TMA bounds; 0 = unknown) */
  int32_t cin, cout, kvol;
  const int32_t* nbr;      /* (kvol, cap_out) */
  const uint32_t* tile_mask;
  int32_t cap_out;
  const int32_t* d_n_out;
  const void* w;           /* f32 (kvol,cin,cout) | packed 16-bit */
  const float* bias;       /* (cout) folded BN */
  const void* residual;    /* (cap_out, cout) same dtype as out, nullable */
  int32_t relu;
  void* out;               /* (cap_out, cout) */
  int32_t out_dtype;
  float* dense;            /* nullable */
  const int32_t* out_coors;
  int32_t out_dims[4];
} srf_conv_args;
int srf_spconv_f32(const srf_conv_args* a_host, void* stream);
int srf_spconv_tc(const srf_conv_args* a_host, void* stream);
int srf_spconv_bf16(const srf_conv_args* a_host, void* stream);
/* w_f32 (kvol, cin, cout) device -> packed 16-bit elements (kvol*cin*cout, twice that for the
 * split encodings) in the order the kernel's shared-memory tiles use */
int srf_pack_weight_tc(const float* w_f32, int32_t kvol, int32_t cin, int32_t cout, int32_t enc,
                       void* w_packed, void* stream);
int srf_pack_weight_bf16(const float* w_f32, int32_t kvol, int32_t cin, int32_t cout, void* w_packed,
                         void* stream);
/* f32 rows -> rows of c_pad (>= c, zero padded) elements in a 16-bit encoding (split rows are
 * [hi(c_pad) | lo(c_pad)]).  srf_f32_to_bf16: the SRF_BF16 form. */
int srf_convert_rows(const float* in, int64_t rows, int32_t c, int32_t c_pad, int32_t enc, void* out,
                     void* stream);
int srf_f32_to_bf16(const float* in, int64_t rows, int32_t c, int32_t c_pad, void* out, void* stream);

/* ---------------------------------------------------------------------------------- *
 * Dense linear on tcgen05: out = epi(A (m,k) . W(n,k)^T + bias).  Replaces the cuBLAS
 * GEMMs of DynamicConv (srfdet_head.py:2668,2689) and the fusion projection (:2257-2262).
 * A bf16 row-major, W packed by srf_pack_linear_bf16 from nn.Linear's (n,k) f32 weight.
 * epi: bit0 relu, bit1 layernorm over n (requires n == tile n <= 128) with ln_w/ln_b.
 * k multiple of 16 (and of 128 when k > 128); n multiple of 16 (of 128 when n > 128).
 * k_splits > 1 (few output tiles, long K, e.g. DynamicConv.out_layer 900x6272x128): the K
 * slices are dealt to k_splits CTAs per tile; split s writes its fp32 partial to slab s of
 * `out` (k_splits, m, n); epi must be 0 and bias NULL.  srf_layernorm(n_partials=k_splits) sums
 * the slabs in order (deterministic) and applies bias/LN/ReLU.  The effective split count is
 * ceil(kvol / ceil(kvol / k_splits)) with kvol = k / min(k,128) (srf_linear_splits).
 * ---------------------------------------------------------------------------------- */
/* srf_linear_tc: A (m,k) in a 16-bit encoding a_enc (plain or split), W packed by
 * srf_pack_linear_tc for the same encoding, out in out_enc (SRF_F32 or a 16-bit form of A's
 * element format), LayerNorm eps explicit, optional residual (m, n) in out's encoding added before
 * the LayerNorm (norm(x + linear(y)) rows of the head: srfdet_head.py:2286-2287, 2304-2306).  K slices are min(k,128) wide (64 for split operands:
 * srf_linear_tile_k_enc).  The *_bf16 / un-suffixed functions are the SRF_BF16, eps = 1e-5 forms. */
int srf_linear_tile_k_enc(int32_t k, int32_t enc);
int srf_linear_splits_enc(int32_t k, int32_t enc, int32_t k_splits);
int srf_pack_linear_tc(const float* w_f32, int32_t n, int32_t k, int32_t enc, void* w_packed, void* stream);
int srf_linear_tc(const void* a, int32_t a_enc, int32_t m, int32_t k, const void* w_packed, int32_t n,
                  const float* bias, const void* residual, int32_t epi, const float* ln_w, const float* ln_b,
                  float ln_eps, void* out, int32_t out_enc, int32_t k_splits, void* stream);
/* The same through an argument block, with the options the head's stage tail uses: A read through a row stride
 * (a column block of a wider buffer), a second copy of the result in another encoding (fp32 trunk + 16-bit GEMM
 * operand from one epilogue), one LayerNorm per 128-column tile (cls | reg towers merged into one GEMM). */
typedef struct srf_linear_args {
  const void* a;        /* (m, k) in a_enc */
  int32_t a_enc, m, k;
  int64_t a_stride;     /* elements between rows of A; 0 = k (2k for split encodings) */
  int64_t a_lo_off;     /* split encodings: elements from a row's hi part to its lo part; 0 = k */
  const void* w;        /* packed by srf_pack_linear_tc */
  int32_t n;
  const float* bias;    /* (n) nullable */
  const void* residual; /* (m, n) in out_enc, nullable */
  int32_t epi;          /* bit0 relu, bit1 layernorm */
  const float *ln_w, *ln_b;
  float ln_eps;
  int32_t ln_per_tile;  /* 1: ln_w / ln_b are (n) and every 128-column tile is normalised on its own */
  void* out;
  int32_t out_enc;
  void* out2;           /* nullable: (m, n) second copy in out2_enc */
  int32_t out2_enc;
  int32_t k_splits;
} srf_linear_args;
int srf_linear(const srf_linear_args* args_host, void* stream);
int srf_linear_tile_k(int32_t k); /* host: K-slice width used by the packer (min(k,128)) */
int srf_linear_tile_n(int32_t n); /* host: N tile width (min(n,128)) */
int srf_linear_splits(int32_t k, int32_t k_splits); /* host: effective split count used for (k, k_splits) */
int srf_pack_linear_bf16(const float* w_f32, int32_t n, int32_t k, void* w_packed, void* stream);
int srf_linear_bf16(const void* a_bf16, int32_t m, int32_t k, const void* w_packed, int32_t n,
                    const float* bias, int32_t epi, const float* ln_w, const float* ln_b,
                    void* out, int32_t out_dtype, int32_t k_splits, void* stream);

/* FP32-mode linear (SIMT FFMA): out = relu?(A (m,k) . W(n,k)^T + bias), any n, k. */
int srf_linear_f32(const float* a, int32_t m, int32_t k, const float* w, int32_t n, const float* bias,
                   int32_t relu, float* out, void* stream);
/* Row-wise LayerNorm (+ReLU) of (sum_p x[p] + bias) over (rows, n); `in` holds n_partials slabs
 * of (rows, n) (split-K partials, summed in slab order; 1 = plain); bias nullable; dtype SRF_F32 | SRF_BF16.
 * Used where the norm cannot be fused into a GEMM epilogue (n > 128, FP32 mode). */
int srf_layernorm(const void* in, int32_t dtype, int64_t rows, int32_t n, int32_t n_partials,
                  const float* bias, const float* gamma, const float* beta, float eps, int32_t relu,
                  void* out, void* stream);
/* same with separate encodings (in f32 | bf16 | f16, out any SRF_* encoding) and an optional f32
 * residual (rows, n) added before the norm: out = act(LN(sum_p in[p] + bias + residual)); out2 (nullable):
 * a second copy of the result in out2_enc (fp32 trunk + 16-bit GEMM operand from one pass) */
int srf_layernorm_enc(const void* in, int32_t in_enc, int64_t rows, int32_t n, int32_t n_partials,
                      const float* bias, const float* residual, const float* gamma, const float* beta, float eps,
                      int32_t relu, void* out, int32_t out_enc, void* out2, int32_t out2_enc, void* stream);

/* ---------------------------------------------------------------------------------- *
 * Region features.
 * srf_boxes_to_corners: boxes3d_to_corners3d(bottom_center=False, ry=False)
 *   (core/bbox/util.py:84-176).  boxes (nb, box_dim>=8) -> corners (nb, 8, 3).
 * ---------------------------------------------------------------------------------- */
int srf_boxes_to_corners(const float* boxes, int32_t nb, int32_t box_dim, float* corners, void* stream);

typedef struct srf_pyramid {
  const float* feat[4]; /* level l: (n_img, C, H_l, W_l) f32 NCHW */
  int32_t h[4], w[4];
  float stride[4];      /* featmap_strides */
  int32_t n_levels;     /* pooler.num_inputs */
  int32_t channels;
  int32_t channels_last; /* 1: maps are (n_img, H_l, W_l, C) in memory (torch.channels_last tensors, C % 4 == 0) */
} srf_pyramid;

/* Generic SingleRoIExtractor + RoIAlign(7x7, sampling_ratio 2, avg, aligned): replaces
 * mmdet SingleRoIExtractor.forward / mmcv roi_align_forward
 * (srfdet_head.py:1685,2082,2548,2626).  rois (k,5) = (img_idx, x1,y1,x2,y2).
 * out (k, C, 7, 7) when channel_last == 0, else (k, 49, C). */
int srf_roi_extract(const srf_pyramid* p_host, const float* rois, int32_t k, float* out,
                    int32_t channel_last, void* stream);

/* Destination of the fused samplers.  channel_last = 0: (k, C, 7, 7) f32 (reference layout).
 * channel_last = 1: rows (k*49 + bin) of row_stride elements (0 -> C, 2C for split encodings),
 * written at channel offset ch_offset, dtype = any SRF_* encoding -- so the image and BEV samplers
 * can fill the two halves of the concatenated fusion input (srfdet_head.py:2257) directly, in the
 * GEMM's encoding.  Split encodings: the row is [hi(row_stride/2) | lo(row_stride/2)] and ch_offset
 * applies inside each half.  16-bit / strided forms need torch.channels_last feature maps. */
typedef struct srf_roi_out {
  void* ptr;
  int32_t channel_last;
  int32_t dtype;
  int32_t row_stride;
  int32_t ch_offset;
} srf_roi_out;

/* Fused points_feats_sampling_bboxes_roi (srfdet_head.py:2568-2629 / 1627-1688):
 * centre de-normalisation IN PLACE on `boxes` (:2587) when mutate != 0, corners, BEV
 * rectangle, level map, RoIAlign.  boxes (B, P, box_dim).  Maps are (B, C, H_l, W_l).
 * out as in srf_roi_extract (k = B*P).  rois_out (B*P,5) nullable (for parity checks). */
int srf_bev_roi_features(const srf_pyramid* p_host, float* boxes, int32_t batch, int32_t n_prop,
                         int32_t box_dim, const float pc_range_host[6], const float voxel_size_host[3],
                         int32_t mutate, const srf_roi_out* out_host, float* rois_out, void* stream);

/* Fused img_feats_sampling_bboxes_roi (srfdet_head.py:2424-2565 / 1963-2099) over a batch of
 * B independent samples, each with the batch-1 semantics of SURVEY.md 3.4 (the reference itself is
 * only defined at B = 1): projection by its own lidar2img[b] (n_cam,4,4), per-camera rectangle,
 * level map, RoIAlign, sum over that sample's cameras in registers.  Maps are
 * (B*n_cam, C, H_l, W_l) (NCHW or channels_last); image b*n_cam + cam is camera cam of sample b.
 * boxes (B, P, box_dim) normalised centres, NOT mutated.  lidar2img (B, n_cam, 4, 4).  Output row
 * k = b*P + p (as in srf_roi_extract, every srf_roi_out form).  rois_out (B*n_cam*P, 5) nullable:
 * row (b*n_cam + cam)*P + p, column 0 = b*n_cam + cam, the image index srf_roi_extract reads.
 * batch < 1 is SRF_ERR_ARG. */
int srf_img_roi_features(const srf_pyramid* p_host, const float* boxes, int32_t batch, int32_t n_prop, int32_t box_dim,
                         const float* lidar2img, int32_t n_cam, const float pc_range_host[6],
                         const srf_roi_out* out_host, float* rois_out, void* stream);

/* DynamicConv interaction core (srfdet_head.py:2679-2686): per proposal
 *   f = relu(LN_d(feats(49,C) . P1(C,d))) ; g = relu(LN_C(f . P2(d,C)))
 * roi (K,49,C) f32|bf16, params (K, 2*C*d) f32|bf16 (P1 then P2, row-major),
 * out (K, 49*C) f32|bf16 (dtype flags).  C <= 256, d <= 64.
 * srf_dynconv_interact_tc: explicit LayerNorm eps and every encoding: a 16-bit out_enc selects the
 * mma.sync kernel ((C,d) = (128,32) | (256,64)) in that element format; roi f32, that format, or
 * (split out) the same split form; params f32 or (plain out) that format; split out rows are
 * [hi(49*C) | lo(49*C)], i.e. the A operand of srf_linear_tc. */
int srf_dynconv_interact_tc(const void* roi, int32_t roi_enc, const void* params, int32_t param_enc,
                            int32_t k, int32_t c, int32_t d, const float* ln1_w, const float* ln1_b,
                            float ln1_eps, const float* ln2_w, const float* ln2_b, float ln2_eps,
                            void* out, int32_t out_enc, void* stream);
int srf_dynconv_interact(const void* roi, int32_t roi_dtype, const void* params, int32_t param_dtype,
                         int32_t k, int32_t c, int32_t d, const float* ln1_w, const float* ln1_b,
                         const float* ln2_w, const float* ln2_b, void* out, int32_t out_dtype,
                         void* stream);

/* ---------------------------------------------------------------------------------- *
 * Rest of a head stage, proposal generation and decoding (SURVEY.md 8f ranks 2, 3), fp32.
 * ---------------------------------------------------------------------------------- */
/* nn.MultiheadAttention core of self_attn_lidar (srfdet_head.py:2281-2285): qkv (B*P, 3*H*hd) f32 =
 * in_proj output (q | k | v), rows batch-major; out (B*P, H*hd) = softmax(q k^T / sqrt(hd)) v per
 * (batch, head), in any encoding (A operand of the out_proj GEMM).  hd in {8,16,32}. */
int srf_mha_attention(const float* qkv, int32_t n_batch, int32_t n_p, int32_t n_heads, int32_t head_dim,
                      void* out, int32_t out_enc, void* stream);
/* SingleSRFDetHead.apply_deltas_lidar (srfdet_head.py:2331-2420): deltas (k,dim), boxes (k,dim) with
 * ABSOLUTE centres and log sizes, weights (dim) device -> out (k,dim) normalised centres, log sizes. */
int srf_apply_deltas(const float* deltas, const float* boxes, int32_t k, int32_t dim, const float* weights,
                     float scale_clamp, const float pc_range_host[6], float* out, void* stream);
/* A (n, c, h, w) map read through element strides: NCHW or torch.channels_last tensors in place. */
typedef struct srf_map {
  const float* ptr;
  int32_t c;
  int64_t sn, sc, sh, sw;
} srf_map;
/* DPG staircase step (srfdet_head.py:521-533; mmcv ConvModule = depthwise Conv2d(3, s2, p1, bias=False) +
 * BN2d(eval, folded) + ReLU) over cat(a, b) (b nullable): out (n, ca+cb, ho, wo) f32, NCHW or
 * (channels_last_out) (n, ho, wo, ca+cb) in memory. */
int srf_dwconv3x3_s2(const srf_map* a_host, const srf_map* b_host, int32_t n, int32_t h, int32_t w,
                     const float* wt_folded, const float* bias_folded, int32_t relu, int32_t channels_last_out,
                     float* out, void* stream);
/* pfeat_34.sum(dim=1) over cat(a, b) (:534); group > 1 / (ho,wo) != (h,w): the image branch's nearest
 * F.interpolate + sum over the cameras of a sample (:584-590).  out (n_samples, ho*wo). */
int srf_channel_sum(const srf_map* a_host, const srf_map* b_host, int32_t n_samples, int32_t group, int32_t h,
                    int32_t w, int32_t ho, int32_t wo, float* out, void* stream);
/* out (m,n) = act(x (m,k) . W (n,k)^T + bias), 1 <= m <= 524280 rows (dpg_fc1 / dpg_fc2, :537-543; one row per
 * sample).  Rows run in groups of 8, one launch; each row is bit-identical to a call with that row alone. */
int srf_gemv_f32(const float* x, int32_t m, int32_t k, const float* w, int32_t n, const float* bias,
                 int32_t relu, float* out, void* stream);
/* (logits_a (+ logits_b)/2) (B,E,P) -> softmax over E -> boxes (B,P,dim) = sum_e w emb_boxes[e,p] with the
 * sigmoid of the centre coordinates (:403, when sigmoid_centres) and feats (B,P,c) = sum_e w emb_feats[e,p]
 * (:597-640) */
int srf_dpg_mix(const float* logits_a, const float* logits_b, int32_t n_batch, int32_t n_exp, int32_t n_p,
                const float* emb_boxes, int32_t box_dim, const float* emb_feats, int32_t c, float* boxes,
                float* feats, int32_t sigmoid_centres, void* stream);
/* get_bboxes decode (:1245-1268 + core/bbox/util.py:41-81): scores = sigmoid(logits) (n_logits values);
 * boxes (k,dim) [abs centre, log size, sin, cos (, vx, vy)] -> out (k,dim-1) [cx, cy, cz - h/2, w, l, h,
 * atan2(sin,cos) (, vx, vy)] */
int srf_decode_boxes(const float* logits, int64_t n_logits, const float* boxes, int32_t k, int32_t dim,
                     float* scores, float* out, void* stream);

/* ---------------------------------------------------------------------------------- *
 * BEV NMS of SRFDetHead.get_bboxes with test_cfg.use_nms=True (sparse_heads/srfdet_head.py:1269-1296:
 * xywhr2xyxyr -> mmdet3d box3d_multiclass_nms -> mmcv nms_bev / nms_normal_bev).  csrc/nms_bev.cu.
 * Footprint of a box row: centre (x, y), extent dx along (cos yaw, sin yaw), dy along (-sin yaw, cos yaw).
 * IoU = inter / (area a + area b - inter), 0 when an area is < 1e-14; suppression is IoU > iou_thr. */
/* pairwise BEV IoU; box rows of width lda/ldb >= 7 with x, y, dx, dy, yaw at columns 0, 1, 3, 4, 6; rotated = 0: axis-aligned
 * dx x dy (yaw ignored).  iou (m, n) row-major. */
int srf_iou_bev(const float* a, int32_t m, int32_t lda, const float* b, int32_t n, int32_t ldb, int32_t rotated, float* iou, void* stream);
size_t srf_nms_bev_ws_bytes(int32_t bs, int32_t k, int32_t n_cls);
/* multi-class BEV NMS of get_bboxes; boxes (bs, k, dim >= 7), scores (bs, k, n_cls); post_center_range: host values passed into the kernel
 * arguments like srf_apply_deltas' pc_range, NULL = no filter.  Per sample and class c: candidates scores[:, c] > score_thr in
 * (score desc, index asc) order, greedy NMS; the kept lists are concatenated class-major; above max_num the max_num best scores are
 * kept in (score desc, class-major position asc) order; then the range filter on columns 0..2 (order preserved).  Outputs of
 * capacity max_num per sample: out_boxes (bs, max_num, dim), out_scores / out_labels (class) / out_index (row in boxes)
 * (bs, max_num), d_count (bs); rows past the count hold a zero box, score 0, label and index -1.  k <= 1024, n_cls <= 32
 * (SRF_ERR_UNSUPPORTED otherwise).  3 launches, no host synchronisation. */
int srf_nms_bev(const float* boxes, int32_t bs, int32_t k, int32_t dim, const float* scores, int32_t n_cls, float score_thr,
                float iou_thr, int32_t rotated, int32_t max_num, const float post_center_range[6], void* ws, size_t ws_bytes,
                float* out_boxes, float* out_scores, int32_t* out_labels, int32_t* out_index, int32_t* d_count, void* stream);

/* ---------------------------------------------------------------------------------- *
 * Multi-sweep point input (mmdet3d 1.0.0rc6 LoadPointsFromMultiSweeps + PointsRangeFilter): the key frame and its
 * sweeps merged into one fixed-capacity cloud.  Source s holds cap rows of ld floats at `points` (device), of which
 * the first clamp(d_counts[s], 0, cap) are points.  In source order, then row order, a point is dropped when
 * SRF_SWEEP_REMOVE_CLOSE and |x| < close_radius and |y| < close_radius (raw values), or when range_host (host
 * values, NULL = none) is given and not lo < p < hi on x, y, z (after the transform).  SRF_SWEEP_TRANSFORM:
 * xyz = fl32(fl32(R xyz) + t) in float64 with numpy's rounding (R row-major then t: d_poses[s][12]);
 * SRF_SWEEP_TIME_LAG: column 4 becomes d_lags[s].  Kept points are written, columns cols_host[0..n_cols) of the
 * modified row, to consecutive rows of out (sum cap, n_cols); *d_total = their number; rows past it are NaN, which
 * every voxelizer drops as out of range.  2 launches, no allocation, no host synchronisation: a captured call
 * replays with new counts, poses and lags.
 * ---------------------------------------------------------------------------------- */
#define SRF_SWEEP_MAX_SOURCES 64
#define SRF_SWEEP_MAX_COLS 8
#define SRF_SWEEP_TRANSFORM 1
#define SRF_SWEEP_TIME_LAG 2
#define SRF_SWEEP_REMOVE_CLOSE 4
typedef struct srf_sweep_src {
  const float* points;
  int32_t cap;
  int32_t ld;
  int32_t flags;
} srf_sweep_src;
size_t srf_merge_sweeps_ws_bytes(const srf_sweep_src* srcs_host, int32_t n_src);
int srf_merge_sweeps(const srf_sweep_src* srcs_host, int32_t n_src, const int32_t* d_counts, const double* d_poses,
                     const float* d_lags, const int32_t* cols_host, int32_t n_cols, const float range_host[6],
                     float close_radius, float* out, int32_t* d_total, void* ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------------- *
 * Test-time augmentation (mmdet3d 1.0.0rc6 MultiScaleFlipAug3D around GlobalRotScaleTrans and RandomFlip3D, with
 * merge_aug_bboxes_3d).  csrc/augment.cu, csrc/nms_bev.cu.  A view is (scale, flips): flip bit SRF_AUG_FLIP_HORIZONTAL
 * negates y, SRF_AUG_FLIP_VERTICAL negates x.  Both entries take the workspace as (ws, *ws_bytes): ws = NULL stores the
 * size they need in *ws_bytes and returns, without touching anything else.
 * ---------------------------------------------------------------------------------- */
#define SRF_AUG_MAX_VIEWS 32
#define SRF_AUG_MAX_COLS 8
#define SRF_AUG_FLIP_HORIZONTAL 1
#define SRF_AUG_FLIP_VERTICAL 2
#define SRF_MERGE_AUG_MAX_K 4096
/* points (cap, n_cols) device, of which the first clamp(*d_count, 0, cap) rows are points (d_count NULL: all cap) ->
 * n_views views out (n_views, cap, n_cols).  Per view a and row, in row order: xyz = fl32(xyz * scales_host[a]), then
 * the flips of flips_host[a]; when range_host (host values, NULL = none) is given, a point is kept only if lo < p < hi
 * on x, y and z (PointsRangeFilter after the augmentation).  Other columns are copied.  Kept rows are compacted stably
 * to the front of their view; d_counts[a] = their number; rows past it are NaN.  2 launches, no allocation, no host
 * synchronisation: a captured call replays with a new count.  3 <= n_cols <= SRF_AUG_MAX_COLS. */
int srf_augment_points(const float* points, int32_t cap, int32_t n_cols, const int32_t* d_count, int32_t n_views,
                       const float* scales_host, const int32_t* flips_host, const float range_host[6], float* out,
                       int32_t* d_counts, void* ws, size_t* ws_bytes, void* stream);
/* merge_aug_bboxes_3d per sample over n_views views of that sample's detections: boxes (bs, n_views, m, dim >= 7)
 * rows [x, y, z, dx, dy, dz, yaw (, vx, vy)], scores (bs, n_views, m), labels (bs, n_views, m) int32, d_counts
 * (bs, n_views): the first clamp(count, 0, m) rows of a view are detections (srf_nms_bev's outputs).  Each row is
 * mapped back (bbox3d_mapping_back, fp32): a horizontal flip negates columns 1::7 then yaw = -yaw; a vertical flip
 * negates columns 0::7 then yaw = fl32(-yaw + fl32(pi)); then every column but yaw is multiplied by
 * inv_scales_host[a] (= fl32(1 / scale)).  The views are concatenated in order; per class (labels outside
 * [0, n_cls) take no part) a greedy NMS in (score desc, concatenated position asc) order suppresses a box whose BEV
 * IoU (srf_iou_bev; rotated = 0: axis-aligned) with a kept one is > iou_thr; the kept lists are concatenated
 * class-major and sorted by (score desc, class-major position asc); the first min(max_num, total) are written.
 * Outputs of capacity max_num per sample: out_boxes (bs, max_num, dim), out_scores, out_labels (bs, max_num), d_count
 * (bs); rows past the count hold a zero box, score 0 and label -1.  n_views * m <= SRF_MERGE_AUG_MAX_K,
 * n_views <= SRF_AUG_MAX_VIEWS and n_cls <= 32 (SRF_ERR_UNSUPPORTED otherwise).  4 launches, no host
 * synchronisation. */
int srf_merge_aug_bev(const float* boxes, const float* scores, const int32_t* labels, const int32_t* d_counts, int32_t bs,
                      int32_t n_views, int32_t m, int32_t dim, const float* inv_scales_host, const int32_t* flips_host,
                      int32_t n_cls, float iou_thr, int32_t rotated, int32_t max_num, void* ws, size_t* ws_bytes,
                      float* out_boxes, float* out_scores, int32_t* out_labels, int32_t* d_count, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SRFDET_B200_H_ */
