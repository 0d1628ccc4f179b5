// Implicit gather-GEMM on tcgen05 / TMEM (sm_100a): the tensor-core modes of the sparse
// convolution (SURVEY.md 8 row a5) and of the dense projections of the region-fusion
// head (rows a9, a10).
//
//   out[m, :] = epi( sum_k  A[idx_k(m), k-slice] . W_k  + bias )
//
// sparse conv : idx_k(m) = nbr[k][m] (rulebook, -1 -> zero row), k-slice = whole row
// dense linear: idx_k(m) = m, k-slice = columns [k*CIN, (k+1)*CIN)
//
// Operand precision (include/srfdet_b200.h):
//   SRF_F16 / SRF_BF16   one tcgen05.mma per 16 input channels (kind::f16, fp32 accumulate)
//   SRF_F16X2 / SRF_BF16X2 ("split", the tensor-core form of the reference's FP32 mode): every
//     value is stored as hi + lo (two 16-bit elements), rows are [hi | lo], weights likewise, and
//     each 16-channel step issues three MMAs  Al.Wh + Ah.Wl + Ah.Wh  into the same fp32
//     accumulator: products are exact to ~2^-16 (bf16) / 2^-21 (f16) relative.
// The operand format (bf16 / f16) is a run-time field of the instruction descriptor; the split
// form is a template parameter because it changes the shared-memory geometry.
//
// Output-stationary: one CTA owns a 128-row output tile; the 128xCOUT fp32 accumulator
// lives in TMEM (double buffered so the epilogue of tile i overlaps the main loop of tile
// i+1) and is written exactly once with bias / residual / ReLU / LayerNorm fused.
//
// Warp roles (4 + NPW + 1 warps; NPW = 4 gather warps, 8 when a slot row is 256 bytes):
//   warps 0-3        epilogue  : tcgen05.ld (warp w owns TMEM lanes 32w..32w+31 = rows), fused
//                                epilogue, global stores
//   warps 4..4+NPW-1 producers : 16-byte cp.async row pieces, consecutive lanes on consecutive
//                                pieces of one row (zero-fill for missing neighbours), + the W_k
//                                tile by cp.async.bulk, into a STAGES-deep mbarrier ring; the
//                                neighbour indices are prefetched one tile ahead (registers ->
//                                shared memory) and read one ring slot ahead
//   last warp        MMA       : one elected lane issues tcgen05.mma (M=128, N=COUT, K=16) per 16
//                                input channels; tcgen05.commit releases ring slots / publishes
//                                the accumulator
// A ring slot carries KC input channels of G kernel offsets (KC = CIN, or CIN/2 when a split row
// would not fit: the offset is then fed as KSPL = 2 consecutive slots reusing the same indices).
// The measured reasons for each of these choices are in profiles/r01_notes.md, r02_notes.md.
// The gather goes through cp.async (row indices are data dependent and -1 rows must read
// zeros; a TMA gather4 variant was correct but 2x slower, tools/variants/) into the canonical
// no-swizzle K-major core-matrix layout:
//   operand byte offset(row r, 16B chunk c) = c * LBO + r * 16     (SBO = 128)
// Launched with programmatic stream serialization: the prologue (barriers, TMEM, resident
// weights) overlaps the tail of the previous kernel, griddepcontrol.wait precedes the first
// access to activations.
#include "igemm_common.cuh"

namespace srf {
// Per-role cycle counters (development builds only: -DSRF_IGEMM_PROF, tools/igemm_prof.py)
#ifdef SRF_IGEMM_PROF
__device__ unsigned long long g_prof[1024 * 16];
__device__ unsigned long long g_prof_t[64 * 1024 * 4];   // [launch % 64][cta] globaltimer: CTA start, main loop start, CTA end
__device__ __forceinline__ unsigned long long gtimer() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#define PROF_T(slot_) if (threadIdx.x == 0) g_prof_t[(((a.dbg >> 16) & 63) * 1024 + (blockIdx.x & 1023)) * 4 + (slot_)] = gtimer()
// event trace of CTA 0 of every launch: (code << 56 | globaltimer); codes: 1 idx publish begin, 2 publish end,
// 3 slots of the tile issued, 4 MMA tile begin, 5 MMA tile committed, 6 epilogue begin, 7 epilogue end
__device__ unsigned long long g_trace[64 * 256];
__device__ int g_trace_n[64];
#define PROF_TRACE(code_) do { if (blockIdx.x == 0) { const int l_ = (a.dbg >> 16) & 63; const int i_ = atomicAdd(&g_trace_n[l_], 1); if (i_ < 256) g_trace[l_ * 256 + i_] = ((unsigned long long)(code_) << 56) | (gtimer() & 0x00ffffffffffffffull); } } while (0)
#define PROF_TBEGIN(v_) v_ -= clock64()
#define PROF_TEND(v_) v_ += clock64()
#if SRF_IGEMM_PROF >= 2      // per-stage cycle counters (perturb the loops by ~200 clk per slot)
#define PROF_DECL(v_) long long v_ = 0
#define PROF_BEGIN(v_) v_ -= clock64()
#define PROF_END(v_) v_ += clock64()
#else
#define PROF_DECL(v_) long long v_ = 0
#define PROF_BEGIN(v_)
#define PROF_END(v_)
#endif
#define PROF_STORE(slot_, v_) g_prof[(blockIdx.x & 1023) * 16 + (slot_)] = (unsigned long long)(v_)
#else
#define PROF_DECL(v_)
#define PROF_BEGIN(v_)
#define PROF_END(v_)
#define PROF_STORE(slot_, v_)
#define PROF_T(slot_)
#define PROF_TBEGIN(v_)
#define PROF_TEND(v_)
#define PROF_TRACE(code_)
#endif

// ring depth cap, and one-CTA-per-SM deep-ring layouts for narrow / 64-channel rows (A/B knobs)
#ifndef SRF_IGEMM_MAXSTAGES
#define SRF_IGEMM_MAXSTAGES 8
#endif
#ifndef SRF_IGEMM_BIG_NARROW
#define SRF_IGEMM_BIG_NARROW 0
#endif
#ifndef SRF_IGEMM_BIG_64
#define SRF_IGEMM_BIG_64 0
#endif
// largest weight set (KB) kept resident in shared memory for rows of <= 4 chunks (A/B knob: 0 = always stream W_k per slot,
// which frees the space for a deeper ring)
#ifndef SRF_IGEMM_WRES_KB
#define SRF_IGEMM_WRES_KB 56
#endif
// resident CTAs per SM aimed at for rows of <= 4 chunks (2 or 3; 3 = 74 KB of smem and <= 72 registers per thread)
#ifndef SRF_IGEMM_CTAS_NARROW
#define SRF_IGEMM_CTAS_NARROW 2
#endif
// gather warps per CTA for rows of <= 4 / 8 / 16 chunks (A/B knobs)
#ifndef SRF_IGEMM_NPW_NARROW
#define SRF_IGEMM_NPW_NARROW 4
#endif
#ifndef SRF_IGEMM_NPW_64
#define SRF_IGEMM_NPW_64 4
#endif
#ifndef SRF_IGEMM_NPW_128
#define SRF_IGEMM_NPW_128 8
#endif

#ifdef SRF_IGEMM_PROF
#define DBG(bit_) (a.dbg & (bit_))
#else
#define DBG(bit_) false
#endif
// input channels per ring slot of split operands with 64 / 128 input channels (A/B knobs)
#ifndef SRF_SPLIT_KC64
#define SRF_SPLIT_KC64 32
#endif
#ifndef SRF_SPLIT_KC128
#define SRF_SPLIT_KC128 64
#endif
// input channels per ring slot of PLAIN 16-bit operands with >= 128 input channels in the sparse form (A/B knob: 64 halves the
// slot so that two CTAs fit per SM)
#ifndef SRF_KC128
#define SRF_KC128 128
#endif

template <int CIN, int COUT, bool SPARSE, bool SPLIT>
struct Cfg {
  // input channels carried by one slot member; an offset takes KSPL consecutive slots
  static constexpr int KC = !SPLIT ? ((SPARSE && CIN >= 128) ? SRF_KC128 : (CIN > 128 ? 128 : CIN))
                                   : (CIN == 64 ? (SPARSE ? SRF_SPLIT_KC64 : 64) : (CIN >= 128 ? SRF_SPLIT_KC128 : CIN));
  static constexpr int KSPL = CIN / KC;
  static constexpr int NJ = KC / 16;                     // MMA K-steps per member (x3 when split)
  static constexpr int CH = (SPLIT ? 2 : 1) * KC / 8;    // 16-byte chunks per A row per slot member (hi planes, then lo planes)
  // For 16 input channels one ring slot carries G kernel offsets (128-byte slot rows): the fixed
  // per-slot cost of the ring (~0.4 us per slot) is then paid once per 64 channels.
  // (measured: 16-channel layers -15 %; at Cin = 32 the doubled slot leaves too few slots in 104 KB)
  static constexpr bool TRI = SPARSE && CH <= 4 && SRF_IGEMM_CTAS_NARROW == 3;   // three CTAs per SM
  static constexpr int G = (SPARSE && CIN == 16) ? ((TRI || SPLIT) ? 2 : 4) : 1;
  // gather warps per CTA (measured, profiles/r01_notes.md): 4 for slot rows <= 128 B (two CTAs per SM),
  // 8 for 256-byte rows (one CTA per SM); the chunked epilogue keeps the register budget low
  static constexpr int NPW = SPARSE ? (CH >= 16 ? SRF_IGEMM_NPW_128 : (CH >= 8 ? SRF_IGEMM_NPW_64 : SRF_IGEMM_NPW_NARROW)) : 4;
  static constexpr int NPT = NPW * 32;
  static constexpr int THREADS = 32 * (4 + NPW + 1);
  static constexpr int MMA_WARP = 4 + NPW;
  static constexpr int PPT = CH * 128 / NPT;  // 16-byte pieces per producer thread per slot member
  static constexpr int A_PAD = CH == 2 ? 64 : (CH == 4 ? 32 : 16);
  static constexpr int A_LBO = 128 * 16 + A_PAD;
  static constexpr int A_MEMBER = CH * A_LBO;
  static constexpr int A_BYTES = G * A_MEMBER;
  static constexpr int B_LBO = COUT * 16;
  static constexpr int B_MEMBER = CH * B_LBO;            // [hi planes | lo planes] of KC x COUT
  // tiny weight sets stay resident in shared memory; otherwise W_k arrives by bulk copy
  static constexpr bool WRES = SPARSE && KSPL == 1 && (27 * B_MEMBER <= (TRI ? 16 : (CH <= 4 ? (SPLIT ? 28 : SRF_IGEMM_WRES_KB) : 16)) * 1024);
  static constexpr int W_BYTES = WRES ? (27 * B_MEMBER + 127) / 128 * 128 : 0;
  static constexpr int B_BYTES = WRES ? 0 : G * B_MEMBER;
  static constexpr int IDX_BYTES = SPARSE ? 27 * 128 * 4 : 0;   // neighbour indices of the current tile
  static constexpr int STAGE_BYTES = (A_BYTES + B_BYTES + 127) / 128 * 128;
  static constexpr bool BIG = SPARSE && ((CH <= 4 && SRF_IGEMM_BIG_NARROW) || (CH == 8 && SRF_IGEMM_BIG_64));   // one CTA per SM, deep ring
  static constexpr int NEED3 = STAGE_BYTES * 3 + W_BYTES + IDX_BYTES;        // three ring slots
  static constexpr bool TWO_WIDE = SPARSE && SRF_KC128 < 128 && NEED3 > 100 * 1024 && NEED3 <= 113 * 1024 - 512;   // knob: 2 CTAs/SM x 3 slots for 128-wide tiles
  static constexpr int BUDGET = TRI ? 73 * 1024 : (TWO_WIDE ? NEED3 + 256 : ((BIG || NEED3 > 100 * 1024) ? 222 * 1024 : 104 * 1024));
  static constexpr int STAGES_RAW = (BUDGET - W_BYTES - IDX_BYTES) / STAGE_BYTES;
  static constexpr int STAGES = STAGES_RAW > SRF_IGEMM_MAXSTAGES ? SRF_IGEMM_MAXSTAGES : (STAGES_RAW < 2 ? 2 : STAGES_RAW);
  static constexpr int TMEM_COLS = 2 * COUT < 32 ? 32 : 2 * COUT;
  static constexpr int BAR_BYTES = (2 * STAGES + 4) * 8 + 16 + (SPARSE ? 0 : 3 * 128 * 4);   // + the dense epilogue's staged bias | ln_w | ln_b
  static constexpr int SMEM_BYTES = W_BYTES + IDX_BYTES + STAGES * STAGE_BYTES + BAR_BYTES + 128;
  static constexpr int MINB = (TRI && COUT <= 64) ? 3 : (((SMEM_BYTES <= 110 * 1024 && COUT <= 64) || TWO_WIDE) ? 2 : 1);
  // kind::f16: D fp32 (bit 4), A/B format at bits 7 / 10 (0 = f16, 1 = bf16: set at run time), K-major both, N>>3 @17, M>>4 @24
  static constexpr uint32_t IDESC0 = (1u << 4) | ((uint32_t)(COUT >> 3) << 17) | ((128u >> 4) << 24);
};

// next group of up to G active kernel offsets from the remaining-offset bit mask
template <int G>
struct Group {
  int n;
  int k[G];
};
template <int G>
__device__ __forceinline__ Group<G> pop_group(uint64_t& rem) {
  Group<G> g;
  g.n = 0;
#pragma unroll
  for (int i = 0; i < G; ++i) {
    g.k[i] = 0;
    if (rem) {
      g.k[i] = __ffsll((long long)rem) - 1;
      rem &= rem - 1;
      g.n = i + 1;
    }
  }
  return g;
}

template <int CIN, int COUT, bool SPARSE, bool SPLIT>
__global__ void __launch_bounds__(Cfg<CIN, COUT, SPARSE, SPLIT>::THREADS, Cfg<CIN, COUT, SPARSE, SPLIT>::MINB)
igemm_umma_kernel(const IgemmArgs a) {
  using C = Cfg<CIN, COUT, SPARSE, SPLIT>;
  constexpr int S = C::STAGES;
  constexpr int G = C::G;
  constexpr int KSPL = C::KSPL;
  static_assert(SPARSE || KSPL == 1, "dense K slices are never sub-split");
  extern __shared__ __align__(128) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 127) & ~(uintptr_t)127);
  uint8_t* w_res = smem;
  int32_t* idx_s = reinterpret_cast<int32_t*>(smem + C::W_BYTES);   // [27][128]
  uint8_t* stage_base = smem + C::W_BYTES + C::IDX_BYTES;
  uint64_t* bars = (uint64_t*)(stage_base + S * C::STAGE_BYTES);
  uint32_t* tmem_slot = (uint32_t*)(bars + 2 * S + 4);
  float* epi_par = reinterpret_cast<float*>(tmem_slot + 4);          // dense form: 3 x 128 floats (16-byte aligned)
  const uint32_t bar0 = smem_u32(bars);
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (S + s); };
  auto tfull_bar = [&](int b) { return bar0 + 8u * (2 * S + b); };
  auto tempty_bar = [&](int b) { return bar0 + 8u * (2 * S + 2 + b); };

  PROF_T(0);
  pdl_trigger();   // the next kernel on the stream may start its own prologue
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_rows = SPARSE ? (a.d_n_out ? min(*a.d_n_out, a.cap_out) : a.cap_out) : a.m_rows;
  const int m_tiles = (m_rows + 127) >> 7;
  const int ksp = SPARSE ? 1 : max(a.k_splits, 1);
  const int kper = (a.kvol + ksp - 1) / ksp;   // K slices per split
  const int mn_tiles = m_tiles * a.n_tiles;
  const int total_tiles = mn_tiles * ksp;
  const uint64_t all_k = a.kvol >= 64 ? ~0ull : ((1ull << a.kvol) - 1ull);

  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) { mbar_init(full_bar(s), ((SPARSE && DBG(128)) ? C::NPW : C::NPT) + (C::WRES ? 0 : 1)); mbar_init(empty_bar(s), 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(tfull_bar(b), 1); mbar_init(tempty_bar(b), 128); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == C::MMA_WARP) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)C::TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (C::WRES) {
    // resident weights: packed global image == shared image ([k][hi|lo][KC/8][COUT][8])
    const uint4* wsrc = reinterpret_cast<const uint4*>(a.w);
    uint4* wdst = reinterpret_cast<uint4*>(w_res);
    const int n16 = a.kvol * (C::B_MEMBER / 16);
    for (int j = threadIdx.x; j < n16; j += blockDim.x) wdst[j] = __ldg(wsrc + j);
    fence_proxy_async();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  // (the OR-reduction is a no-op on the value: it tells the compiler the address is warp-uniform,
  // which keeps the MMA issue sequence free of per-instruction broadcast loops)
  const uint32_t tmem_base = __reduce_or_sync(0xffffffffu, *tmem_slot);
  const uint32_t stage_u32 = smem_u32(stage_base), wres_u32 = smem_u32(w_res);
  PROF_T(1);
  // everything above (barriers, TMEM, resident weights) is independent of the previous kernel;
  // activations, residuals and every global write come after this point
  pdl_wait();

  if (warp >= 4 && warp < 4 + C::NPW) {
    // ------------------------------------------------------------------ producers
    const int pt = threadIdx.x - 128;
    int it = 0;
    // Neighbour indices: thread pt prefetches the 27 indices of row pt one tile ahead into
    // registers (27 independent loads in flight), then publishes them to shared memory at
    // the tile boundary, because the copy mapping below spreads a row over several lanes.
    int cur[27];
    uint32_t mask = 0xffffffffu;
    auto load_idx = [&](int tile) {
      mask = 0xffffffffu;
      if (!SPARSE) return;
      const bool live = tile < total_tiles;
      const int mt = live ? tile % m_tiles : 0;
      const int row = mt * 128 + pt;
      if (a.tile_mask) mask = live ? __ldg(a.tile_mask + mt) : 0u;
#pragma unroll
      for (int k = 0; k < 27; ++k) {
        cur[k] = -1;
        if (live && pt < 128 && k < a.kvol && ((mask >> k) & 1u) && row < m_rows) cur[k] = __ldg(a.nbr + (size_t)k * a.cap_out + row);
      }
    };
    PROF_DECL(p_total); PROF_DECL(p_empty); PROF_DECL(p_pub); PROF_DECL(p_issue); PROF_DECL(p_arr); PROF_DECL(p_fetch);
    PROF_TBEGIN(p_total);
    load_idx(blockIdx.x);
    // copy mapping: the 128*CH 16-byte pieces of a slot member are dealt out so that consecutive
    // lanes take consecutive pieces of the SAME row (coalesced: a warp instruction touches
    // 32/CH rows x one contiguous row segment each instead of 32 different rows; measured
    // 2.4x the LDGSTS rate of the thread-per-row mapping for 64-byte rows, tools/micro/).
    // Thread pt always copies chunk c = pt % CH of rows r0 + i * RSTEP; chunks [0, CH/2) of a
    // split row come from its hi part, the rest from its lo part.
    constexpr int CHS = C::CH == 2 ? 1 : (C::CH == 4 ? 2 : (C::CH == 8 ? 3 : 4));
    static_assert(C::CH == 2 || C::CH == 4 || C::CH == 8 || C::CH == 16, "slot rows of 32..256 bytes");
    constexpr int RSTEP = C::NPT / C::CH;
    const int pc = pt & (C::CH - 1), r0 = pt >> CHS;
    const uint32_t dst_off = (uint32_t)(pc * C::A_LBO + r0 * 16);
    const long long pcol = (SPLIT && pc >= C::CH / 2) ? a.in_lo_off + (pc - C::CH / 2) * 8 : (long long)pc * 8;   // elements
    const char* src_c = reinterpret_cast<const char*>(a.in + pcol);
    const uint32_t row_bytes = (uint32_t)(a.in_stride * 2);
    // idx_s[k][r0 * PPT + i] = neighbour index of row r0 + i * RSTEP: the PPT indices a thread
    // needs for one slot are adjacent, one vector LDS fetches them
    const uint32_t idx_s_addr = smem_u32(idx_s) + (uint32_t)(r0 * C::PPT) * 4u;
    const int pub_pos = (pt % RSTEP) * C::PPT + pt / RSTEP;   // where row pt's index goes
    int gi[G][C::PPT];   // neighbour indices of this thread's rows for the (up to G) offsets of the slot being filled
    // shared-memory index reads are issued one slot AHEAD (right after the copies of the
    // current slot): an LDS queues behind every LDGSTS already in the LSU pipe, and a
    // load -> copy -> load -> copy chain exposed that queueing delay once per piece.
    auto fetch_one = [&](int* g, int k) {
      const uint32_t ad = idx_s_addr + (uint32_t)(k * 128 * 4);
      if constexpr (C::PPT == 1) {
        asm volatile("ld.shared.b32 %0, [%1];" : "=r"(g[0]) : "r"(ad));
      } else if constexpr (C::PPT == 2) {
        asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(g[0]), "=r"(g[1]) : "r"(ad));
      } else {
#pragma unroll
        for (int i = 0; i < C::PPT; i += 4)
          asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(g[i]), "=r"(g[i + 1]), "=r"(g[i + 2]), "=r"(g[i + 3]) : "r"(ad + i * 4));
      }
    };
    // indices of the next (up to G) active offsets, without consuming them
    auto fetch_idx = [&](uint32_t rem) {
      if (DBG(16)) return;
#pragma unroll
      for (int m = 0; m < G; ++m) {
        if (rem) fetch_one(gi[m], __ffs((int)rem) - 1);
        rem &= rem - 1;
      }
    };
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const int mt = tile % m_tiles, nt = (tile % mn_tiles) / m_tiles, ks = tile / mn_tiles;
      uint32_t tmask = mask;
      if (SPARSE) {
        if (pt == 0) PROF_TRACE(1);
        PROF_BEGIN(p_pub);
        asm volatile("bar.sync 1, %0;" ::"n"(C::NPT) : "memory");   // previous tile's indices no longer read
        if (pt < 128) {
#pragma unroll
          for (int k = 0; k < 27; ++k) idx_s[k * 128 + pub_pos] = cur[k];
        }
        asm volatile("bar.sync 1, %0;" ::"n"(C::NPT) : "memory");
        PROF_END(p_pub);
        if (pt == 0) PROF_TRACE(2);
        load_idx(tile + gridDim.x);                       // next tile's indices, in flight during the fills
        uint32_t rem = tmask & (uint32_t)all_k;
        fetch_idx(rem);
        while (rem) {
          int kk[G], n = 0;
#pragma unroll
          for (int m = 0; m < G; ++m) {
            kk[m] = 0;
            if (rem) { kk[m] = __ffs((int)rem) - 1; rem &= rem - 1; n = m + 1; }
          }
#pragma unroll
          for (int q = 0; q < KSPL; ++q) {
            const int s = it % S;
            const uint32_t ph = (uint32_t)(it / S) & 1u;
            PROF_BEGIN(p_empty);
            if (!DBG(512)) mbar_wait(empty_bar(s), ph ^ 1u);
            PROF_END(p_empty);
            const uint32_t sa = smem_u32(stage_base + s * C::STAGE_BYTES);
            PROF_BEGIN(p_issue);
            if (!DBG(1)) {
#pragma unroll
              for (int m = 0; m < G; ++m) {
                if (m < n) {
#pragma unroll
                  for (int i = 0; i < C::PPT; ++i) {
                    const int src_row = gi[m][i];
                    const char* src = src_c + (size_t)(uint32_t)max(src_row, 0) * row_bytes + q * (C::KC * 2);
                    cp_async16_ca(sa + (uint32_t)(m * C::A_MEMBER) + dst_off + (uint32_t)(i * RSTEP * 16), src, src_row >= 0 ? 16u : 0u);
                  }
                }
              }
            }
            PROF_END(p_issue);
            PROF_BEGIN(p_arr);
            if (!C::WRES && pt == 0) {
              // the W_k tiles (packed global image == shared image) arrive by bulk copy (UBLKCP),
              // tracked by the same barrier through its transaction count
              const uint32_t fb = full_bar(s);
              if (DBG(2)) {
                asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(fb) : "memory");
              } else {
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(fb), "r"((uint32_t)(n * C::B_MEMBER)) : "memory");
#pragma unroll
                for (int m = 0; m < G; ++m)
                  if (m < n)
                    bulk_g2s(sa + C::A_BYTES + m * C::B_MEMBER,
                             a.w + (((size_t)nt * a.kvol + kk[m]) * KSPL + q) * (size_t)(C::B_MEMBER / 2), C::B_MEMBER, fb);
              }
            }
            // the hardware arrives on full[s] for this thread when its copies have landed
            // (cutlass::arch::cpasync_barrier_arrive_noinc pattern): producers never wait on data
            if (DBG(512)) {}
            else if (DBG(128)) { __syncwarp(); if (lane == 0) mbar_arrive(full_bar(s)); }
            else if (DBG(64)) mbar_arrive(full_bar(s));
            else asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(full_bar(s)) : "memory");
            PROF_END(p_arr);
            ++it;
          }
          PROF_BEGIN(p_fetch);
          fetch_idx(rem);
          PROF_END(p_fetch);
        }
        if (pt == 0) PROF_TRACE(3);
      } else {
        // dense linear: every K slice of this split, in order (kvol may exceed 64); rows are
        // the tile's own, no index traffic at all
        for (int k = ks * kper; k < min(a.kvol, (ks + 1) * kper); ++k) {
          const int s = it % S;
          const uint32_t ph = (uint32_t)(it / S) & 1u;
          mbar_wait(empty_bar(s), ph ^ 1u);
          const uint32_t sa = smem_u32(stage_base + s * C::STAGE_BYTES);
#pragma unroll
          for (int i = 0; i < C::PPT; ++i) {
            const int r = r0 + i * RSTEP;
            const bool ok = mt * 128 + r < m_rows;
            const uint16_t* src = ok ? a.in + (size_t)(mt * 128 + r) * a.in_stride + (size_t)k * a.k_stride + pcol : a.in;
            cp_async16_ca(sa + dst_off + (uint32_t)(i * RSTEP * 16), src, ok ? 16u : 0u);
          }
          if (pt == 0) {
            const uint32_t fb = full_bar(s);
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(fb), "r"((uint32_t)C::B_MEMBER) : "memory");
            bulk_g2s(sa + C::A_BYTES, a.w + ((size_t)nt * a.kvol + k) * (size_t)(C::B_MEMBER / 2), C::B_MEMBER, fb);
          }
          asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(full_bar(s)) : "memory");
          ++it;
        }
      }
    }
    PROF_TEND(p_total);
    if (pt == 0) { PROF_STORE(0, p_total); PROF_STORE(1, p_empty); PROF_STORE(2, p_pub); PROF_STORE(3, it); PROF_STORE(11, p_issue); PROF_STORE(12, p_arr); PROF_STORE(13, p_fetch); }
    asm volatile("cp.async.wait_all;" ::: "memory");
  } else if (warp == C::MMA_WARP) {
    // ------------------------------------------------------------------ MMA issuer
    int it = 0, tcount = 0;
    const uint32_t idesc = C::IDESC0 | (a.fmt ? 0u : ((1u << 7) | (1u << 10)));
    PROF_DECL(m_total); PROF_DECL(m_full); PROF_DECL(m_tempty); PROF_DECL(m_issue);
    PROF_TBEGIN(m_total);
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++tcount) {
      const int mt = tile % m_tiles;
      const uint32_t mask = (SPARSE && a.tile_mask) ? __ldg(a.tile_mask + mt) : 0xffffffffu;
      const int buf = tcount & 1;
      const uint32_t tph = (uint32_t)(tcount >> 1) & 1u;
      if (lane == 0) PROF_TRACE(4);
      PROF_BEGIN(m_tempty);
      mbar_wait(tempty_bar(buf), tph ^ 1u);
      PROF_END(m_tempty);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + (uint32_t)(buf * COUT);
      uint32_t accumulate = 0;
      uint64_t rem = SPARSE ? ((uint64_t)mask & all_k) : 0ull;
      int kd = (tile / mn_tiles) * kper;             // dense linear: K-slice counter of this split
      const int kd_end = min(a.kvol, (tile / mn_tiles + 1) * kper);
      while (SPARSE ? (rem != 0) : (kd < kd_end)) {
        Group<G> g;
        if (SPARSE) {
          g = pop_group<G>(rem);
        } else {
          g.n = 1;
          g.k[0] = kd++;
        }
#pragma unroll
        for (int q = 0; q < KSPL; ++q) {
          const int s = it % S;
          const uint32_t ph = (uint32_t)(it / S) & 1u;
          PROF_BEGIN(m_full);
          if (!DBG(512)) mbar_wait(full_bar(s), ph);
          PROF_END(m_full);
          tc_fence_after();
          PROF_BEGIN(m_issue);
          {
            // descriptors advance additively (start-address field += bytes >> 4): one uniform add per MMA
            const uint32_t sa = stage_u32 + (uint32_t)s * C::STAGE_BYTES;
            const uint32_t a_lo0 = ((sa >> 4) & 0x3fffu) | ((uint32_t)(C::A_LBO >> 4) << 16);
            const uint32_t b_lo0 = (((sa + C::A_BYTES) >> 4) & 0x3fffu) | ((uint32_t)(C::B_LBO >> 4) << 16);
            const uint32_t w_lo0 = ((wres_u32 >> 4) & 0x3fffu) | ((uint32_t)(C::B_LBO >> 4) << 16);
            if (elect_one_sync()) {
#pragma unroll
              for (int m = 0; m < G; ++m) {
                if (m < g.n) {
                  const uint32_t a_lo = a_lo0 + (uint32_t)(m * (C::A_MEMBER >> 4));
                  const uint32_t b_lo = C::WRES ? w_lo0 + (uint32_t)g.k[m] * (uint32_t)(C::B_MEMBER >> 4) : b_lo0 + (uint32_t)(m * (C::B_MEMBER >> 4));
#pragma unroll
                  for (int j = 0; j < C::NJ; ++j) {
                    const uint64_t ah = desc_pack(a_lo + (uint32_t)(j * ((2 * C::A_LBO) >> 4)), DESC_HI);
                    const uint64_t bh = desc_pack(b_lo + (uint32_t)(j * ((2 * C::B_LBO) >> 4)), DESC_HI);
                    if (SPLIT) {
                      // hi/lo planes: [0, NJ) hi, [NJ, 2 NJ) lo.  Small cross terms first, then the main product.
                      const uint64_t al = desc_pack(a_lo + (uint32_t)((C::NJ + j) * ((2 * C::A_LBO) >> 4)), DESC_HI);
                      const uint64_t bl = desc_pack(b_lo + (uint32_t)((C::NJ + j) * ((2 * C::B_LBO) >> 4)), DESC_HI);
                      if (!DBG(4)) {
                        tc_mma_f16(tmem_d, al, bh, idesc, accumulate);
                        tc_mma_f16(tmem_d, ah, bl, idesc, 1u);
                        tc_mma_f16(tmem_d, ah, bh, idesc, 1u);
                      }
                    } else {
                      if (!DBG(4)) tc_mma_f16(tmem_d, ah, bh, idesc, accumulate);
                    }
                    accumulate = 1;
                  }
                }
              }
              if (DBG(512)) {} else if (DBG(32)) mbar_arrive(empty_bar(s)); else tc_commit(empty_bar(s));
            }
          }
          PROF_END(m_issue);
          __syncwarp();
          accumulate = 1;
          ++it;
        }
      }
      if (elect_one_sync()) tc_commit(tfull_bar(buf));
      __syncwarp();
      if (lane == 0) PROF_TRACE(5);
    }
    PROF_TEND(m_total);
    if (lane == 0) { PROF_STORE(4, m_total); PROF_STORE(5, m_full); PROF_STORE(6, m_tempty); PROF_STORE(7, tcount); PROF_STORE(14, m_issue); }
  } else {
    // ------------------------------------------------------------------ epilogue
    int tcount = 0;
    PROF_DECL(e_total); PROF_DECL(e_tfull);
    PROF_TBEGIN(e_total);
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++tcount) {
      const int mt = tile % m_tiles, nt = (tile % mn_tiles) / m_tiles;
      const int buf = tcount & 1;
      const uint32_t tph = (uint32_t)(tcount >> 1) & 1u;
      PROF_BEGIN(e_tfull);
      mbar_wait(tfull_bar(buf), tph);
      PROF_END(e_tfull);
      if (threadIdx.x == 0) PROF_TRACE(6);
      tc_fence_after();
      const int row = mt * 128 + warp * 32 + lane;
      const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(buf * COUT);
      if (SPARSE) {
        // a tile whose mask has no active offset got no MMA, and its TMEM buffer still holds an older tile's
        // accumulator (or uninitialised TMEM): its rows are act(bias + residual), so the sum is zero here
        const bool no_mma = a.tile_mask && (((uint64_t)__ldg(a.tile_mask + mt) & all_k) == 0ull);
        // drain the accumulator in 32-column chunks (small register footprint)
        constexpr int NC = COUT < 32 ? COUT : 32;
#pragma unroll 1
        for (int c0 = 0; c0 < COUT; c0 += NC) {
          float v[NC];
#pragma unroll
          for (int cc = 0; cc < NC; cc += 16) tc_ld16(taddr + c0 + cc, v + cc);
          if (no_mma) {
#pragma unroll
            for (int c = 0; c < NC; ++c) v[c] = 0.f;
          }
          if (row < m_rows && !DBG(8)) epilogue_chunk<COUT, NC>(a, row, nt * COUT + c0, v);
        }
        tc_fence_before();
        mbar_arrive(tempty_bar(buf));
      } else {
        // stage the tile's epilogue parameters (the 4 epilogue warps = threads 0..127; COUT <= 128)
        asm volatile("bar.sync 2, 128;" ::: "memory");      // the previous tile's parameters are no longer read
        if ((int)threadIdx.x < COUT && a.k_splits <= 1) {
          const int col = nt * COUT + threadIdx.x;
          epi_par[threadIdx.x] = a.bias ? __ldg(a.bias + col) : 0.f;
          epi_par[128 + threadIdx.x] = a.ln ? __ldg(a.ln_w + (a.ln_per_tile ? col : (int)threadIdx.x)) : 1.f;
          epi_par[256 + threadIdx.x] = a.ln ? __ldg(a.ln_b + (a.ln_per_tile ? col : (int)threadIdx.x)) : 0.f;
        }
        asm volatile("bar.sync 2, 128;" ::: "memory");
        float v[COUT];
#pragma unroll
        for (int c0 = 0; c0 < COUT; c0 += 16) tc_ld16(taddr + c0, v + c0);
        // accumulator is in registers: hand the TMEM buffer back to the MMA warp
        tc_fence_before();
        mbar_arrive(tempty_bar(buf));
        if (row < m_rows && !DBG(8)) epilogue_row<COUT>(a, row, nt, v, epi_par, tile / mn_tiles);
      }
      if (threadIdx.x == 0) PROF_TRACE(7);
    }
    PROF_TEND(e_total);
    if (threadIdx.x == 0) { PROF_STORE(8, e_total); PROF_STORE(9, e_tfull); PROF_STORE(10, gridDim.x); }
  }
  tc_fence_before();
  __syncthreads();
  PROF_T(2);
  if (warp == C::MMA_WARP) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)C::TMEM_COLS) : "memory");
  }
}

#ifdef SRF_IGEMM_PROF
static int g_prof_launch = 0;
static int prof_next_launch() { return g_prof_launch++; }
static int prof_dbg_env() { const char* e = getenv("SRF_IGEMM_DBG"); return e ? atoi(e) : 0; }
#endif

template <int CIN, int COUT, bool SPARSE, bool SPLIT>
static int launch_igemm(const IgemmArgs& a, int host_tiles, cudaStream_t st) {
  using C = Cfg<CIN, COUT, SPARSE, SPLIT>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(igemm_umma_kernel<CIN, COUT, SPARSE, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES);
    if (e != cudaSuccess) { set_error("igemm<%d,%d>: cannot set %d B dynamic smem: %s", CIN, COUT, C::SMEM_BYTES, cudaGetErrorString(e)); return SRF_ERR_CUDA; }
    configured = true;
  }
  int per_sm = (227 * 1024) / (C::SMEM_BYTES + 1024);
  int by_tmem = 512 / C::TMEM_COLS;
  if (per_sm > by_tmem) per_sm = by_tmem;
  if (per_sm > C::MINB) per_sm = C::MINB;
  if (per_sm < 1) per_sm = 1;
  int grid = sm_count() * per_sm;
  if (grid > host_tiles) grid = host_tiles;
  if (grid < 1) grid = 1;
  SRF_COUNT(1);
  IgemmArgs ap = a;
#ifdef SRF_IGEMM_PROF
  ap.dbg = prof_dbg_env() | ((prof_next_launch() & 63) << 16);
#endif
  cudaError_t e = launch_pdl(igemm_umma_kernel<CIN, COUT, SPARSE, SPLIT>, dim3(grid), dim3(C::THREADS), (size_t)C::SMEM_BYTES, st, ap);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("igemm<%d,%d> launch failed: %s", CIN, COUT, cudaGetErrorString(e)); return SRF_ERR_CUDA; }
  return SRF_OK;
}

// NOTE: a window-staged mma.sync form of the 32 -> 32 / 16 -> 16 layers (contiguous input windows in shared memory, ldmatrix
// gathers) is parity-green but instruction-bound at 98 vs 77 us (profiles/r02_notes.md; tools/variants/spconv_window.cu.txt).
// Two other producers were built and measured slower on B200 (profiles/r01_notes.md): the TMA
// tile::gather4 form (~45 clk per 4-row instruction, ~2x slower; archived in tools/variants/) and a
// register-staged LDG -> STS form (1.5x slower).  Neither is part of the build.

// channel pairs of the encoders of the four configs (SURVEY.md Appendix A) plus the head's tiles
template <bool SPLIT>
static int dispatch_sparse(int cin, int cout, const IgemmArgs& a, int host_tiles, cudaStream_t st) {
#define SRF_CASE(ci, co) if (cin == ci && cout == co) return launch_igemm<ci, co, true, SPLIT>(a, host_tiles, st);
  SRF_CASE(16, 16) SRF_CASE(16, 32) SRF_CASE(32, 32) SRF_CASE(32, 64) SRF_CASE(64, 64) SRF_CASE(64, 128)
  SRF_CASE(128, 128) SRF_CASE(128, 64) SRF_CASE(64, 32) SRF_CASE(32, 16) SRF_CASE(256, 128) SRF_CASE(256, 64)
#undef SRF_CASE
  set_error("sparse igemm: unsupported channel pair cin=%d cout tile=%d", cin, cout);
  return SRF_ERR_UNSUPPORTED;
}

template <bool SPLIT>
static int dispatch_dense(int tk, int tn, const IgemmArgs& a, int host_tiles, cudaStream_t st) {
  // (split operands use K slices of at most 64 channels: srf_linear_tile_k_enc)
#define SRF_CASE(ci, co) if constexpr (!(SPLIT && ci > 64)) { if (tk == ci && tn == co) return launch_igemm<ci, co, false, SPLIT>(a, host_tiles, st); }
  SRF_CASE(128, 128) SRF_CASE(64, 128) SRF_CASE(32, 128) SRF_CASE(16, 128)
  SRF_CASE(128, 64) SRF_CASE(64, 64) SRF_CASE(32, 64) SRF_CASE(16, 64)
  SRF_CASE(128, 32) SRF_CASE(64, 32) SRF_CASE(32, 32) SRF_CASE(16, 32)
  SRF_CASE(128, 16) SRF_CASE(64, 16) SRF_CASE(32, 16) SRF_CASE(16, 16)
#undef SRF_CASE
  set_error("dense igemm: unsupported tile k=%d n=%d", tk, tn);
  return SRF_ERR_UNSUPPORTED;
}

}  // namespace srf

using namespace srf;

#ifdef SRF_IGEMM_PROF
extern "C" int srf_prof_read(unsigned long long* host, int reset) {
  cudaDeviceSynchronize();
  if (host) cudaMemcpyFromSymbol(host, srf::g_prof, sizeof(srf::g_prof));
  if (reset) { static unsigned long long z[1024 * 16]; cudaMemcpyToSymbol(srf::g_prof, z, sizeof(z)); }
  return 0;
}
extern "C" int srf_prof_trace(unsigned long long* host, int launch) {   // host[256]; returns the number of events
  cudaDeviceSynchronize();
  int n = 0;
  cudaMemcpyFromSymbol(&n, srf::g_trace_n, 4, (size_t)(launch & 63) * 4);
  cudaMemcpyFromSymbol(host, srf::g_trace, 256 * 8, (size_t)(launch & 63) * 256 * 8);
  int z = 0;
  cudaMemcpyToSymbol(srf::g_trace_n, &z, 4, (size_t)(launch & 63) * 4);
  return n < 256 ? n : 256;
}
extern "C" int srf_prof_read_t(unsigned long long* host, int launch) {   // launch < 0: next launch id
  if (launch < 0) return srf::g_prof_launch;
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(host, srf::g_prof_t, 1024 * 4 * 8, (size_t)(launch & 63) * 1024 * 4 * 8);
  return 0;
}
#endif

extern "C" {

int srf_conv_tile_n(int32_t cout);

static bool use_warp16() {
  static int on = -1;
  if (on < 0) { const char* e = getenv("SRF_CONV16_WARP"); on = (e && e[0] == '0') ? 0 : 1; }
  return on != 0;
}

int srf_spconv_tc(const srf_conv_args* c, void* stream) {
  SRF_CHECK_ARG(c && c->in && c->nbr && c->w && (c->out || c->dense), "srf_spconv_tc: null arg");
  SRF_CHECK_ARG(enc_is_16(c->in_dtype), "srf_spconv_tc: input features must be bf16 / f16 / split");
  SRF_CHECK_ARG(c->kvol >= 1 && c->kvol <= 27, "srf_spconv_tc: kvol must be in [1,27]");
  SRF_CHECK_ARG(c->cap_out > 0 && c->cap_out % 128 == 0, "srf_spconv_tc: cap_out must be a multiple of 128");
  SRF_CHECK_ARG(!c->dense || c->out_coors, "srf_spconv_tc: dense output needs out_coors");
  SRF_CHECK_ARG(c->dense || c->out_dtype == SRF_F32 || (enc_is_16(c->out_dtype) && enc_is_f16(c->out_dtype) == enc_is_f16(c->in_dtype)),
                "srf_spconv_tc: a 16-bit output must use the input's element format");
  const bool split = enc_is_split(c->in_dtype);
  // 16 -> 16 channels (the sparsely connected finest level): warp-level MMA kernel, spconv_warp16.cu
  if (!split && c->cin == 16 && c->cout == 16 && c->kvol == 27 && !c->dense && c->out && c->out_dtype == c->in_dtype && use_warp16())
    return spconv16_warp_launch(c, enc_is_f16(c->in_dtype), (cudaStream_t)stream);
  IgemmArgs a = {};
  a.in = (const uint16_t*)c->in;
  a.in_stride = split ? 2 * c->cin : c->cin;
  a.in_lo_off = c->cin;
  a.k_stride = 0;
  a.nbr = c->nbr;
  a.tile_mask = c->tile_mask;
  a.d_n_out = c->d_n_out;
  a.cap_out = c->cap_out;
  a.kvol = c->kvol;
  const int tn = srf_conv_tile_n(c->cout);
  SRF_CHECK_ARG(c->cout % tn == 0 && (tn == c->cout || !c->dense), "srf_spconv_tc: cout > 128 must be a multiple of 128 (and not dense-scattered)");
  a.n_tiles = c->cout / tn;
  a.w = (const uint16_t*)c->w;
  a.bias = c->bias;
  a.residual = c->residual;
  a.relu = c->relu;
  a.out = c->out;
  a.fmt = enc_is_f16(c->in_dtype) ? 1 : 0;
  a.out_enc = c->dense ? SRF_F32 : c->out_dtype;
  a.out_stride = enc_is_split(a.out_enc) ? 2 * c->cout : c->cout;
  a.out_lo_off = c->cout;
  a.dense = c->dense;
  a.out_coors = (const int4*)c->out_coors;
  a.D = c->out_dims[1];
  a.H = c->out_dims[2];
  a.W = c->out_dims[3];
  return split ? dispatch_sparse<true>(c->cin, tn, a, c->cap_out / 128 * a.n_tiles, (cudaStream_t)stream)
               : dispatch_sparse<false>(c->cin, tn, a, c->cap_out / 128 * a.n_tiles, (cudaStream_t)stream);
}

int srf_spconv_bf16(const srf_conv_args* c, void* stream) { return srf_spconv_tc(c, stream); }

// K chunk per ring slot of the sparse kernel (the packer lays the weights out per chunk)
int srf_pack_weight_kc(int32_t cin, int32_t enc) {
  if (!enc_is_split(enc)) return cin >= 128 ? SRF_KC128 : cin;
  return cin == 64 ? SRF_SPLIT_KC64 : (cin >= 128 ? SRF_SPLIT_KC128 : cin);
}
// output-channel tile of the sparse kernel: layers wider than 128 outputs run as cout / 128 column tiles
int srf_conv_tile_n(int32_t cout) { return cout > 128 ? 128 : cout; }

int srf_linear_tile_k_enc(int32_t k, int32_t enc) {
  // K slice per ring slot of the dense tcgen05 GEMM: 128 channels (64 for split operands, whose
  // slot rows carry hi and lo)
  const int cap = enc_is_split(enc) ? 64 : 128;
  return k > cap ? cap : k;
}
int srf_linear_tile_k(int32_t k) { return srf_linear_tile_k_enc(k, SRF_BF16); }
int srf_linear_tile_n(int32_t n) { return n > 128 ? 128 : n; }

int srf_linear_splits_enc(int32_t k, int32_t enc, int32_t k_splits) {
  const int kvol = k / srf_linear_tile_k_enc(k, enc);
  if (k_splits <= 1 || kvol <= 1) return 1;
  const int kper = (kvol + k_splits - 1) / k_splits;
  return (kvol + kper - 1) / kper;
}
int srf_linear_splits(int32_t k, int32_t k_splits) { return srf_linear_splits_enc(k, SRF_BF16, k_splits); }

int srf_linear(const srf_linear_args* p, void* stream) {
  SRF_CHECK_ARG(p, "srf_linear: null args");
  const void* a_in = p->a;
  const int32_t a_enc = p->a_enc, m = p->m, k = p->k, n = p->n, epi = p->epi, out_enc = p->out_enc, k_splits = p->k_splits;
  const void* w_packed = p->w;
  const float *bias = p->bias, *ln_w = p->ln_w, *ln_b = p->ln_b;
  const void* residual = p->residual;
  void* out = p->out;
  const float ln_eps = p->ln_eps;
  SRF_CHECK_ARG(a_in && w_packed && out && m >= 0 && k > 0 && n > 0, "srf_linear_tc: bad args");
  SRF_CHECK_ARG(!p->out2 || p->out2_enc == SRF_F32 || (enc_is_16(p->out2_enc) && enc_is_f16(p->out2_enc) == enc_is_f16(a_enc)),
                "srf_linear_tc: a 16-bit second output must use A's element format");
  SRF_CHECK_ARG(enc_is_16(a_enc), "srf_linear_tc: A must be bf16 / f16 / split");
  SRF_CHECK_ARG(out_enc == SRF_F32 || (enc_is_16(out_enc) && enc_is_f16(out_enc) == enc_is_f16(a_enc)),
                "srf_linear_tc: a 16-bit output must use A's element format");
  if (m == 0) return SRF_OK;
  const bool split = enc_is_split(a_enc);
  int tk = srf_linear_tile_k_enc(k, a_enc), tn = srf_linear_tile_n(n);
  SRF_CHECK_ARG(k % tk == 0 && n % tn == 0, "srf_linear_tc: n=%d k=%d not tileable", n, k);
  SRF_CHECK_ARG(!(epi & 2) || ((n == tn || p->ln_per_tile) && ln_w && ln_b),
                "srf_linear_tc: fused LayerNorm needs n <= 128 (or one norm per 128-column tile) and ln weights");
  IgemmArgs a = {};
  a.in = (const uint16_t*)a_in;
  a.in_stride = p->a_stride > 0 ? p->a_stride : (split ? 2 * k : k);
  a.in_lo_off = p->a_lo_off > 0 ? p->a_lo_off : k;
  a.k_stride = tk;
  a.m_rows = m;
  a.out2 = p->out2;
  a.out2_enc = p->out2_enc;
  a.ln_per_tile = p->ln_per_tile;
  a.cap_out = m;
  a.kvol = k / tk;
  a.n_tiles = n / tn;
  a.w = (const uint16_t*)w_packed;
  a.bias = bias;
  a.residual = residual;
  a.relu = epi & 1;
  a.ln = (epi & 2) ? 1 : 0;
  a.ln_w = ln_w;
  a.ln_b = ln_b;
  a.ln_eps = ln_eps;
  a.out = out;
  a.fmt = enc_is_f16(a_enc) ? 1 : 0;
  a.out_enc = out_enc;
  a.out_stride = enc_is_split(out_enc) ? 2 * n : n;
  a.out_lo_off = n;
  a.k_splits = 1;
  if (k_splits > 1) {
    SRF_CHECK_ARG(epi == 0 && !bias && !residual && !p->out2 && out_enc == SRF_F32,
                  "srf_linear_tc: split-K needs epi=0, no bias / residual / second output and an f32 output of k_splits slabs");
    const int kper = (a.kvol + k_splits - 1) / k_splits;
    a.k_splits = (a.kvol + kper - 1) / kper;   // every split owns at least one K slice
  }
  const int tiles = cdiv(m, 128) * (n / tn) * a.k_splits;
  return split ? dispatch_dense<true>(tk, tn, a, tiles, (cudaStream_t)stream) : dispatch_dense<false>(tk, tn, a, tiles, (cudaStream_t)stream);
}

int srf_linear_tc(const void* a_in, int32_t a_enc, int32_t m, int32_t k, const void* w_packed, int32_t n, const float* bias,
                  const void* residual, int32_t epi, const float* ln_w, const float* ln_b, float ln_eps, void* out, int32_t out_enc,
                  int32_t k_splits, void* stream) {
  srf_linear_args p = {};
  p.a = a_in; p.a_enc = a_enc; p.m = m; p.k = k; p.w = w_packed; p.n = n; p.bias = bias; p.residual = residual; p.epi = epi;
  p.ln_w = ln_w; p.ln_b = ln_b; p.ln_eps = ln_eps; p.out = out; p.out_enc = out_enc; p.k_splits = k_splits;
  return srf_linear(&p, stream);
}

int srf_linear_bf16(const void* a_bf16, int32_t m, int32_t k, const void* w_packed, int32_t n, const float* bias,
                    int32_t epi, const float* ln_w, const float* ln_b, void* out, int32_t out_dtype, int32_t k_splits,
                    void* stream) {
  return srf_linear_tc(a_bf16, SRF_BF16, m, k, w_packed, n, bias, nullptr, epi, ln_w, ln_b, 1e-5f, out, out_dtype, k_splits, stream);
}

}  // extern "C"
