// TDNN affine layer as a tcgen05 GEMM (sm_100a).
//
//   y[b,t,n] = epi( bias[n] + sum_{tap} sum_{c} W[n, tap, c] * x[b, t + ctx[tap], c] )
//
// Restates TdnnAffine.forward + ReLU + eval-BatchNorm of the reference
// (pytorch/libs/nnet/components.py:107-149, :410-431) as ONE kernel:
//   * M = B*T frames, N = Cout, K = ntaps*Cin -- only the taps in `context` (the reference's
//     conv1d also multiplies the masked taps, components.py:133-138);
//   * the context splice is never materialised: the A tile of tap `c` is fetched by TMA from the
//     (C, T, B) frame matrix at time coordinate t0 + c; TMA's out-of-bounds zero fill *is*
//     F.pad(..., value=0) (components.py:117) and can never cross an utterance boundary;
//   * fp32-grade accuracy at bf16 tensor rate: operands are bf16 "split planes" (hi, lo) and each
//     K step issues hi*hi + lo*hi + hi*lo into the same fp32 TMEM accumulator;
//   * warp-specialised persistent CTAs (usually CTA pairs, cta_group::2): warp0 = TMA producer, warp1 =
//     tcgen05.mma issuer, warps2-9 = epilogue (tcgen05.ld -> +bias -> ReLU -> BN -> split -> swizzled smem
//     slab -> TMA store), double-buffered accumulators in TMEM so the epilogue of tile i overlaps the MMAs
//     of tile i+1.
// Variants of the same kernel (template flags): kPool -- swapped operands, the epilogue pools over time
// instead of storing (fused statistics pooling); kHist -- the epilogue bins scores into a trial histogram
// (scoring.cu); runtime: a second A source (W.(a+b)), split-K slices for the segment layers, an im2col
// view of the first layer (x_batch_stride).
//
// An M tile is 128 rows = Bb utterances x Tb consecutive frames (Tb*Bb = 128, chosen on the host
// to minimise padding: T=200 -> Tb=8, Bb=16 has none).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <stdlib.h>

#include <mutex>
#include <type_traits>

#include "common.cuh"
#include "ptx.cuh"

// Timing experiments (profiles/r01_gemm_experiments.md) switch parts of the kernel off and produce
// WRONG results; they exist only when the library is built with -DXVB_TIMING_EXPERIMENTS.
#ifdef XVB_TIMING_EXPERIMENTS
#define XVB_DBG(p, bit) ((p).debug & (bit))
#else
#define XVB_DBG(p, bit) 0
#endif

namespace xvb {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;                      // bf16 elements = one 128-byte swizzle row
constexpr int kABytes = kBlockM * kBlockK * 2;   // 16 KB per plane per stage
constexpr int kNumEpiWarps = 8;                  // two groups of 4 warps, each group covers all 128 TMEM lanes
constexpr int kNumThreads = 64 + kNumEpiWarps * 32;
constexpr int kSlabBytes = 16384;                // TMA-store staging: bf16 hi(8K)+lo(8K) or one fp32 slab
constexpr int kParamBytes = 3 * 256 * 4;         // bias/scale/shift for one 256-wide tile

struct TdnnGemmParams {
  int B, T, Cin, Cout;
  int Tb, Bb, num_t_blk, num_b_blk, num_n_blk, num_tiles;
  int ntaps, cin_p16, num_cblk;
  int ctx[XVB_MAX_TAPS];
  int flags;
  const float* bias;
  const float* scale;
  const float* shift;
  const float* row_bias;  // per-frame additive term (PLDA row term), may be NULL
  const float* utt_bias;  // per-utterance x column additive term (B, ld_utt), may be NULL
  long long ld_utt;
  int log2_tb;            // Tb is a power of two
  int debug;              // -DXVB_TIMING_EXPERIMENTS only: bit0 skip epilogue, bit1 skip MMA, bit2 skip store issue, bit3 skip LDTM,
                          // box64 epilogue: bit4 parameters not read from smem, bit5 slab not filled, bit6 no hand-over barriers
  int plane_box64;        // plane-only outputs: 64-column chunks, hi then lo through the slab, 128-byte store rows
  int store_mode;         // 0: epilogue slab -> TMA store; 1: slab -> coalesced st.global; 2: registers -> st.global (sector-sized)
  float* pool_partial;    // fused statistics pooling: per (time block, utterance, channel) [mean | M2] partials
  int num_src;            // 1, or 2: a second A source accumulated with the same weights (W.(x + x2))
  // M-unit sharding (a unit = kCta x 128 rows): this launch walks units unit_first + k * unit_stride
  int unit_first, unit_stride;
  // fused trial histogram (scoring.cu: xvb_trial_histogram): the scores never leave the SM
  unsigned long long* hist;   // (2, hist_bins) u64 counters [nontarget | target], accumulated; NULL = off
  const int* row_label;       // speaker id per row / per column
  const int* col_label;
  float hist_lo, hist_inv_w;  // bin = 1 + floor((s - lo) * inv_w); bin 0: s < lo; bin nbins-1: at or above hi
  int hist_bins;
  int hist_sym;               // count only column index > row index (all pairs of one set, each once)
  int hist_group, num_units;  // tile raster of the score-matrix mode (decode_tile)
  // split-K for the segment-level layers (M = B rows, K in the thousands: too few tiles to fill the
  // machine otherwise): slice s of a tile covers channel blocks [s*kb_per_slice, (s+1)*kb_per_slice)
  // and stores its fp32 partial at "time" s of a (B, k_slices, Cout) buffer; segment_reduce_kernel sums
  // the slices in order (deterministic) and applies the epilogue.  ntaps == 1, one source only.
  int k_slices, kb_per_slice;
  __nv_bfloat16* y_hi;
  __nv_bfloat16* y_lo;
  long long ldy;
  float* y_f32;
  long long ldyf;
  const int* lengths;     // ragged batch (kMask only): valid frames per utterance, device
};

// kCta = 1: one CTA per 128 x BLOCK_N tile.  kCta = 2: a CTA pair (cluster of 2, tcgen05
// cta_group::2) per 256 x BLOCK_N tile -- each CTA stages its own 128 A rows and HALF of the
// weight tile, so operand traffic per MMA flop drops by a third and a third stage fits.
// kNSub = 2 ("wide"): one tile spans TWO adjacent BLOCK_N column blocks that share the A tile, so the
// frame matrix is fetched once per 512 output channels instead of once per 256 (the operand stream
// out of L2, not the tensor pipe, bounds this kernel: measured 9.2 TB/s with the MMAs skipped).  The
// price: the 512 TMEM columns hold a single accumulator, so the epilogue no longer overlaps the
// next tile's MMAs (its TMA loads still run ahead).
template <int BLOCK_N, int kCta, int kNSub>
struct GemmCfg {
  static constexpr int kBRows = BLOCK_N / kCta;   // weight rows staged by one CTA per column block
  static constexpr int kBBytes = kBRows * kBlockK * 2;          // one plane of one column block
  static constexpr int kStageBytes = 2 * kABytes + 2 * kNSub * kBBytes;
  static constexpr int kStages = (192 * 1024) / kStageBytes > 6 ? 6 : (192 * 1024) / kStageBytes;
  static constexpr int kAccStages = kNSub == 1 ? 2 : 1;
  static constexpr int kTileN = BLOCK_N * kNSub;
  static constexpr int kTmemCols = kAccStages * kTileN < 32 ? 32 : kAccStages * kTileN;
  static_assert(kTmemCols <= 512, "TMEM has 512 columns");
  static constexpr int kSmemBytes =
      kStages * kStageBytes + kSlabBytes + 2 * kParamBytes + 1024 /*align slack*/ + 256 /*barriers*/;
  static_assert(kSmemBytes <= 232448, "exceeds the 227 KB shared memory of an sm_100 CTA");
  static_assert(kStages >= 2, "need at least a double-buffered operand pipeline");
};

// kPool (CTA pairs only): fused statistics pooling.  The MMA operands swap roles -- the weight tile
// is the M side (128 output channels per CTA = TMEM lanes), the frame tile the N side (256 frames =
// TMEM columns) -- so an epilogue thread owns ONE channel and sees the tile's frames as consecutive
// accumulator columns: pooling over time becomes a running (Welford) update in registers, with no
// shuffles, no shared memory and no (B,T,C) output at all.
// Tile index -> (M unit, N block).  Layers: N fastest, so the CTAs running together share the frame
// (A) tile and walk the small, L2-resident weight matrix.  Score matrices (kHist): both operands are
// huge, so tiles are rastered in bands of `hist_group` M units x all N blocks, M fastest -- the ~74
// pairs in flight cover hist_group rows x ~9 columns and each test (B) tile leaves HBM once per band
// instead of once per M unit.  Returns false for tiles that do not exist / lie below the diagonal.
template <bool kHist>
__device__ __forceinline__ bool decode_tile(const TdnnGemmParams& p, int tile, int& m_unit, int& n_blk, int& slice) {
  slice = 0;
  if constexpr (!kHist) {
    if (p.k_slices > 1) { slice = tile % p.k_slices; tile /= p.k_slices; }
    m_unit = p.unit_first + (tile / p.num_n_blk) * p.unit_stride;
    n_blk = tile % p.num_n_blk;
    return true;
  } else {
    const int per_band = p.num_n_blk * p.hist_group;
    const int band = tile / per_band, r = tile - band * per_band;
    n_blk = r / p.hist_group;
    const int mi = band * p.hist_group + (r - n_blk * p.hist_group);
    m_unit = p.unit_first + mi * p.unit_stride;
    return mi < p.num_units && !(p.hist_sym && n_blk < m_unit);
  }
}

// kHist: the epilogue bins the scores into a trial histogram instead of storing them (scoring.cu).
// kMask: ragged batch -- rows t >= lengths[b] store exact zeros (the F.pad zeros the next layer's taps must read) and the
// pooling epilogue counts lengths[b] frames.  A separate instantiation, so the equal-length kernels are untouched.
template <int BLOCK_N, int kCta, int kNSub, bool kPool, bool kHist, bool kMask>
__global__ void __launch_bounds__(kNumThreads, 1)
tdnn_gemm_bf16x3_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                        const __grid_constant__ CUtensorMap map_a2_hi, const __grid_constant__ CUtensorMap map_a2_lo,
                        const __grid_constant__ CUtensorMap map_w_hi, const __grid_constant__ CUtensorMap map_w_lo,
                        const __grid_constant__ CUtensorMap map_y_hi, const __grid_constant__ CUtensorMap map_y_lo,
                        const __grid_constant__ CUtensorMap map_y_f32, const __grid_constant__ TdnnGemmParams p) {
  using Cfg = GemmCfg<BLOCK_N, kCta, kNSub>;
  constexpr int kAccStages = Cfg::kAccStages;
  constexpr int kTileN = Cfg::kTileN;
  constexpr int kStages = Cfg::kStages;
  constexpr int kBBytes = Cfg::kBBytes;
  constexpr int kStageBytes = Cfg::kStageBytes;
  const uint32_t cta_rank = kCta == 2 ? cluster_ctarank() : 0;  // rank 0 = leader (issues the MMAs)
  const int tile_first = kCta == 2 ? blockIdx.x >> 1 : blockIdx.x;
  const int tile_step = kCta == 2 ? gridDim.x >> 1 : gridDim.x;

  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B tiles need 1024-byte alignment
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* slab_base = smem + kStages * kStageBytes;                     // 16 KB, 1024-aligned
  float* param_base = reinterpret_cast<float*>(slab_base + kSlabBytes);  // 2 x [3][256] floats
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(slab_base + kSlabBytes + 2 * kParamBytes);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tmem_full_bar = empty_bar + kStages;
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&map_a_hi);
    tma_prefetch_desc(&map_a_lo);
    tma_prefetch_desc(&map_w_hi);
    tma_prefetch_desc(&map_w_lo);
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&full_bar[i], kCta);   // leader's barrier: one producer arrival per CTA + all TMA bytes
      mbar_init(&empty_bar[i], 1);     // per CTA, released by (multicast) tcgen05.commit
    }
    for (int i = 0; i < kAccStages; ++i) {
      mbar_init(&tmem_full_bar[i], 1);                          // per CTA, (multicast) commit
      mbar_init(&tmem_empty_bar[i], kCta * kNumEpiWarps * 32);  // leader's: every epilogue thread of the pair
    }
    fence_barrier_init();
  }
  if constexpr (kCta == 2) cluster_sync();  // peer barriers initialised before anyone signals them
  if (warp == 1) tmem_alloc<kCta>(tmem_ptr_smem, Cfg::kTmemCols);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  // Programmatic dependent launch: everything above (barrier init, TMEM allocation, descriptor
  // prefetch) may overlap the tail of the previous kernel in the stream; its results are needed from here on.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  // the previous kernel may have written our operands with ordinary (generic-proxy) stores -- the staging
  // / pooling kernels do -- while we read them through TMA (async proxy): order the two proxies explicitly,
  // a kernel boundary would have done it for us
  asm volatile("fence.proxy.async;" ::: "memory");

  const int num_kblk = p.num_src * p.ntaps * p.num_cblk;

  if (warp == 0) {
    // ================================ TMA producer ================================
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = tile_first; tile < p.num_tiles; tile += tile_step) {
        int m_unit, n_blk, slice;
        if (!decode_tile<kHist>(p, tile, m_unit, n_blk, slice)) continue;   // e.g. entirely on or below the diagonal
        const int cb_begin = slice * p.kb_per_slice;                        // (0, num_cblk) unless split-K
        const int cb_end = p.k_slices > 1 ? min(p.num_cblk, cb_begin + p.kb_per_slice) : p.num_cblk;
        const int m_blk = m_unit * kCta + (int)cta_rank;
        const int b0 = (m_blk / p.num_t_blk) * p.Bb, t0 = (m_blk % p.num_t_blk) * p.Tb;  // may be fully out of
        const int n0 = n_blk * kTileN + (int)cta_rank * Cfg::kBRows;                      // range: TMA zero-fills
        for (int src = 0; src < p.num_src; ++src) {
        const CUtensorMap* ma_hi = src == 0 ? &map_a_hi : &map_a2_hi;
        const CUtensorMap* ma_lo = src == 0 ? &map_a_lo : &map_a2_lo;
        for (int tap = 0; tap < p.ntaps; ++tap) {
          const int tt = t0 + p.ctx[tap];
          for (int cb = cb_begin; cb < cb_end; ++cb) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* s = smem + stage * kStageBytes;
            const int kw = tap * p.cin_p16 + cb * kBlockK;
            if constexpr (kCta == 1) {
              mbar_expect_tx(&full_bar[stage], kStageBytes);
              tma_load_3d(s, ma_hi, &full_bar[stage], cb * kBlockK, tt, b0);
              tma_load_3d(s + kABytes, ma_lo, &full_bar[stage], cb * kBlockK, tt, b0);
#pragma unroll
              for (int ns = 0; ns < kNSub; ++ns) {
                tma_load_2d(s + 2 * kABytes + ns * kBBytes, &map_w_hi, &full_bar[stage], kw, n0 + ns * BLOCK_N);
                tma_load_2d(s + 2 * kABytes + (kNSub + ns) * kBBytes, &map_w_lo, &full_bar[stage], kw, n0 + ns * BLOCK_N);
              }
            } else {
              // both CTAs' bytes complete on the LEADER's barrier (peer-bit-masked address)
              if (cta_rank == 0) mbar_expect_tx(&full_bar[stage], 2 * kStageBytes);
              else mbar_arrive_cluster(&full_bar[stage], 0);
              tma_load_3d_2sm(s, ma_hi, &full_bar[stage], cb * kBlockK, tt, b0);
              tma_load_3d_2sm(s + kABytes, ma_lo, &full_bar[stage], cb * kBlockK, tt, b0);
#pragma unroll
              for (int ns = 0; ns < kNSub; ++ns) {
                tma_load_2d_2sm(s + 2 * kABytes + ns * kBBytes, &map_w_hi, &full_bar[stage], kw, n0 + ns * BLOCK_N);
                tma_load_2d_2sm(s + 2 * kABytes + (kNSub + ns) * kBBytes, &map_w_lo, &full_bar[stage], kw, n0 + ns * BLOCK_N);
              }
            }
            if (++stage == kStages) { stage = 0; phase ^= 1; }
          }
        }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ================================ MMA issuer ==================================
    // (leader CTA only: one thread drives the tensor cores of both SMs of a pair)
    if (cta_rank == 0 && elect_one()) {
      constexpr uint32_t idesc = make_idesc_bf16(kBlockM * kCta, BLOCK_N);
      int stage = 0;
      uint32_t phase = 0;
      uint32_t it = 0;
      for (int tile = tile_first; tile < p.num_tiles; tile += tile_step) {
        int kb_begin = 0, kb_end = num_kblk;
        if constexpr (kHist) { int mu, nb, sl; if (!decode_tile<true>(p, tile, mu, nb, sl)) continue; }
        else if (p.k_slices > 1) {
          kb_begin = (tile % p.k_slices) * p.kb_per_slice;
          kb_end = min(num_kblk, kb_begin + p.kb_per_slice);
        }
        const uint32_t acc = kAccStages == 2 ? (it & 1) : 0, acc_phase = kAccStages == 2 ? ((it >> 1) & 1) : (it & 1);
        ++it;
        mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1);
        tcgen05_fence_after();
        const uint32_t tmem_d = tmem_base + acc * kTileN;
        uint32_t accumulate = 0;
        for (int kb = kb_begin; kb < kb_end; ++kb) {
          const int cb = kb % p.num_cblk;
          int nsteps = (p.Cin - cb * kBlockK + 15) >> 4;
          nsteps = nsteps > 4 ? 4 : nsteps;
          mbar_wait(&full_bar[stage], phase);
          tcgen05_fence_after();
          const uint32_t sa = smem_u32(smem + stage * kStageBytes);
          const uint64_t da_hi = make_kmajor_desc<128>(sa);
          const uint64_t da_lo = make_kmajor_desc<128>(sa + kABytes);
          for (int s = 0; s < (XVB_DBG(p, 2) ? 0 : nsteps); ++s) {
            const uint64_t koff = (uint64_t)(s * 32 >> 4);  // 16 bf16 = 32 bytes along K inside the swizzle row
#pragma unroll
            for (int ns = 0; ns < kNSub; ++ns) {
              const uint64_t db_hi = make_kmajor_desc<128>(sa + 2 * kABytes + ns * kBBytes);
              const uint64_t db_lo = make_kmajor_desc<128>(sa + 2 * kABytes + (kNSub + ns) * kBBytes);
              const uint32_t d = tmem_d + ns * BLOCK_N;
              if constexpr (kPool) {  // D^T: channels on the lanes, frames on the columns
                umma_bf16<kCta>(d, db_hi + koff, da_lo + koff, idesc, accumulate);
                umma_bf16<kCta>(d, db_lo + koff, da_hi + koff, idesc, 1);
                umma_bf16<kCta>(d, db_hi + koff, da_hi + koff, idesc, 1);
              } else {
                umma_bf16<kCta>(d, da_lo + koff, db_hi + koff, idesc, accumulate);
                umma_bf16<kCta>(d, da_hi + koff, db_lo + koff, idesc, 1);
                umma_bf16<kCta>(d, da_hi + koff, db_hi + koff, idesc, 1);
              }
            }
            accumulate = 1;
          }
          umma_commit<kCta>(&empty_bar[stage]);  // frees the smem slot (in both CTAs) once these MMAs retire
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit<kCta>(&tmem_full_bar[acc]);  // accumulator complete -> epilogue (of both CTAs)
      }
    }
    __syncwarp();
  } else {
    // ================================ epilogue ====================================
    // 8 warps: warp -> TMEM lane quarter q = warp & 3 (hardware rule) and column half h = (warp-2)>>2;
    // a thread owns one accumulator row and 16 of the 32 columns of every chunk.  Per chunk:
    // tcgen05.ld (prefetched one chunk ahead) -> +bias -> ReLU -> BN (parameters broadcast from
    // smem) -> split -> swizzled 16 KB smem slab -> one thread issues the TMA store, which clips
    // ragged T / B / Cout for free and writes full lines.
    const int ew = warp - 2;
    const int half = ew >> 2;
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int etid = threadIdx.x - 64;  // 0..255
    const bool leader = etid == 0;
    const bool relu = (p.flags & XVB_RELU) != 0;
    const bool bn = (p.flags & XVB_BN) != 0;
    const bool act_sigmoid = (p.flags & XVB_SIGMOID) != 0;
    const bool act_tanh = (p.flags & XVB_TANH) != 0;
    const bool planes = p.y_hi != nullptr;
    const bool f32o = p.y_f32 != nullptr;
    uint32_t it = 0;
    // fused trial histogram: the 16 KB store slab holds 2 x hist_bins u32 counters instead
    constexpr bool hist = kHist;
    uint32_t h_below[2] = {0u, 0u}, h_above[2] = {0u, 0u};   // out-of-window scores: counted in registers
    const uint32_t hslab = smem_u32(slab_base);
    auto hist_flush = [&]() {
      asm volatile("bar.sync 3, 256;" ::: "memory");
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        if (h_below[c]) asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(hslab + (c * p.hist_bins) * 4), "r"(h_below[c]) : "memory");
        if (h_above[c]) asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(hslab + (c * p.hist_bins + p.hist_bins - 1) * 4), "r"(h_above[c]) : "memory");
        h_below[c] = 0u; h_above[c] = 0u;
      }
      asm volatile("bar.sync 3, 256;" ::: "memory");
      for (int e = etid; e < 2 * p.hist_bins; e += kNumEpiWarps * 32) {
        uint32_t c;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(c) : "r"(hslab + e * 4) : "memory");
        if (c) {
          atomicAdd(p.hist + e, (unsigned long long)c);
          asm volatile("st.shared.u32 [%0], %1;" ::"r"(hslab + e * 4), "r"(0u) : "memory");
        }
      }
      asm volatile("bar.sync 3, 256;" ::: "memory");
    };
    if (hist) {
      for (int e = etid; e < 2 * p.hist_bins; e += kNumEpiWarps * 32)
        asm volatile("st.shared.u32 [%0], %1;" ::"r"(hslab + e * 4), "r"(0u) : "memory");
      asm volatile("bar.sync 3, 256;" ::: "memory");
    }
    for (int tile = tile_first; tile < p.num_tiles; tile += tile_step) {
      int m_unit, n_blk, slice;
      if (!decode_tile<kHist>(p, tile, m_unit, n_blk, slice)) continue;
      const uint32_t acc = kAccStages == 2 ? (it & 1) : 0, acc_phase = kAccStages == 2 ? ((it >> 1) & 1) : (it & 1);
      ++it;
      const int m_blk = m_unit * kCta + (int)cta_rank;
      const int b0 = (m_blk / p.num_t_blk) * p.Bb, t0 = (m_blk % p.num_t_blk) * p.Tb;
      const int b = b0 + row / p.Tb, t = t0 + row % p.Tb;
      const bool valid = (b < p.B) && (t < p.T);
      const int n0 = n_blk * kTileN;
      if constexpr (kPool) {
        // ---- fused statistics pooling: thread = channel, accumulator columns = the pair's 256 frames
        const int hb = ew >> 2;                                   // frames of CTA `hb` of the pair (columns hb*128..)
        const int cch = n0 + (int)cta_rank * 128 + q * 32 + lane;  // this thread's output channel
        const bool cvalid = cch < p.Cout;
        const float bias_c = (cvalid && p.bias) ? __ldg(p.bias + cch) : 0.f;
        const float scale_c = (cvalid && bn) ? __ldg(p.scale + cch) : 1.f;
        const float shift_c = (cvalid && bn) ? __ldg(p.shift + cch) : 0.f;
        const float floor_c = relu ? 0.f : -INFINITY;
        const int mh = m_unit * 2 + hb;
        const int bh0 = (mh / p.num_t_blk) * p.Bb, th0 = (mh % p.num_t_blk) * p.Tb, tblk = mh % p.num_t_blk;
        mbar_wait(&tmem_full_bar[acc], acc_phase);
        tcgen05_fence_after();
        const uint32_t tcol = tmem_base + ((uint32_t)(q * 32) << 16) + acc * kTileN + hb * 128;
        float rn = 0.f, rmean = 0.f, rm2 = 0.f;   // running Chan state, only used when a time block spans > 16 columns
        auto emit = [&](int col, float mean, float m2) {
          const int bb = bh0 + (col >> p.log2_tb);
          if (cvalid && bb < p.B) {
            float* dst = p.pool_partial + ((long long)tblk * p.B + bb) * (2LL * p.Cout) + cch;
            dst[0] = mean;
            dst[p.Cout] = m2;
          }
        };
        // one group of G consecutive frame columns (G = min(Tb,16), compile-time): two passes in registers
        auto group = [&](const float* x, int col0, auto gtag) {
          constexpr int G = decltype(gtag)::value;
          const int tt0 = col0 & (p.Tb - 1);
          int len = p.T;
          if constexpr (kMask) {                                   // the group's frames belong to one utterance
            const int bb = bh0 + (col0 >> p.log2_tb);
            len = bb < p.B ? __ldg(p.lengths + bb) : 0;
          }
          int nv = len - (th0 + tt0);                              // valid frames of this group (warp-uniform)
          nv = nv < 0 ? 0 : (nv > G ? G : nv);
          float sum = 0.f;
#pragma unroll
          for (int i = 0; i < G; ++i) sum += i < nv ? x[i] : 0.f;
          const float mean = nv > 0 ? sum / (float)nv : 0.f;
          float m2 = 0.f;
#pragma unroll
          for (int i = 0; i < G; ++i) { const float d = i < nv ? x[i] - mean : 0.f; m2 = fmaf(d, d, m2); }
          if (p.Tb <= 16) {
            if (nv > 0) emit(col0, mean, m2);
          } else {                                                 // Chan merge of 16-frame groups into the block
            if (nv > 0) {
              const float tot = rn + (float)nv, wb = (float)nv / tot, d = mean - rmean;
              rmean = fmaf(d, wb, rmean);
              rm2 += m2 + d * d * rn * wb;
              rn = tot;
            }
            if (tt0 + G == p.Tb) { if (rn > 0.f) emit(col0, rmean, rm2); rn = 0.f; rmean = 0.f; rm2 = 0.f; }
          }
        };
        auto consume = [&](uint32_t (&v)[16], int c16) {
          float x[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) x[j] = fmaf(fmaxf(__uint_as_float(v[j]) + bias_c, floor_c), scale_c, shift_c);
          const int col = c16 * 16;
          switch (p.log2_tb) {
            case 0:
#pragma unroll
              for (int g = 0; g < 16; ++g) group(x + g, col + g, std::integral_constant<int, 1>{});
              break;
            case 1:
#pragma unroll
              for (int g = 0; g < 8; ++g) group(x + 2 * g, col + 2 * g, std::integral_constant<int, 2>{});
              break;
            case 2:
#pragma unroll
              for (int g = 0; g < 4; ++g) group(x + 4 * g, col + 4 * g, std::integral_constant<int, 4>{});
              break;
            case 3:
              group(x, col, std::integral_constant<int, 8>{});
              group(x + 8, col + 8, std::integral_constant<int, 8>{});
              break;
            default:
              group(x, col, std::integral_constant<int, 16>{});
              break;
          }
        };
        uint32_t va[16], vb[16];
        tmem_ld_32x16(tcol, va);
#pragma unroll 1
        for (int c16 = 0; c16 < 8; c16 += 2) {
          tmem_ld_wait();
          tmem_ld_32x16(tcol + (c16 + 1) * 16, vb);
          consume(va, c16);
          tmem_ld_wait();
          if (c16 + 2 < 8) tmem_ld_32x16(tcol + (c16 + 2) * 16, va);
          consume(vb, c16 + 1);
        }
        tcgen05_fence_before();
        if constexpr (kCta == 1) mbar_arrive(&tmem_empty_bar[acc]);
        else mbar_arrive_cluster(&tmem_empty_bar[acc], 0);
        continue;
      }
      bool masked = false;                                 // frame past the end of its utterance: store zeros
      if constexpr (kMask) masked = valid && t >= __ldg(p.lengths + b);
      const float rbias = (p.row_bias && valid) ? __ldg(p.row_bias + (long long)b * p.T + t) : 0.f;
      const float* ub = (p.utt_bias && valid) ? p.utt_bias + (long long)b * p.ld_utt + n0 + half * 16 : nullptr;
      // stage this tile's per-column parameters (double-buffered by accumulator stage; the
      // barrier also orders reuse: nobody can be two tiles ahead of the slowest epilogue thread)
      // layout: kAccStages buffers of [bias | scale | shift], each kTileN floats (6 KB in total either way)
      const uint32_t prm = smem_u32(param_base) + acc * (3 * kTileN * 4);
      if constexpr (kAccStages == 1) asm volatile("bar.sync 3, 256;" ::: "memory");  // single buffer: everyone left the previous tile
      for (int e = etid; e < kTileN; e += kNumEpiWarps * 32) {
        const int c = n0 + e;
        const bool in = c < p.Cout;
        st_shared_f32(prm + e * 4, (in && p.bias) ? __ldg(p.bias + c) : 0.f);
        if (hist) st_shared_f32(prm + (kTileN + e) * 4, __int_as_float(in ? __ldg(p.col_label + c) : -2));
        else st_shared_f32(prm + (kTileN + e) * 4, (in && bn) ? __ldg(p.scale + c) : 1.f);
        st_shared_f32(prm + (2 * kTileN + e) * 4, (in && bn) ? __ldg(p.shift + c) : 0.f);
      }
      asm volatile("bar.sync 3, 256;" ::: "memory");
      int nch = (p.Cout - n0 + 31) >> 5;
      nch = nch > kTileN / 32 ? kTileN / 32 : nch;
      mbar_wait(&tmem_full_bar[acc], acc_phase);
      tcgen05_fence_after();
      const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16) + acc * kTileN + half * 16;
      const uint32_t slab = smem_u32(slab_base);
      const float relu_floor = relu ? 0.f : -INFINITY;   // branch-free ReLU switch
      const bool extras = rbias != 0.f || ub != nullptr || act_tanh || act_sigmoid;
      // TMA stores clip the last 16-byte group of a row as a whole, so in the tile holding column Cout the columns
      // [Cout, round_up(Cout, 16 bytes)) are written too: store zeros there (the pad split_f32 leaves), never epi(0)
      const bool n_tail = n0 + kTileN > p.Cout;

      auto process = [&](uint32_t (&v)[16], int ch) {
        const int pc = ch * 32 + half * 16;
        float f[16];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const float4 bb = ld_shared_f4(prm + (pc + 4 * g) * 4);
          const float4 ss = ld_shared_f4(prm + (kTileN + pc + 4 * g) * 4);
          const float4 tt = ld_shared_f4(prm + (2 * kTileN + pc + 4 * g) * 4);
          float x0 = __uint_as_float(v[4 * g + 0]) + bb.x;
          float x1 = __uint_as_float(v[4 * g + 1]) + bb.y;
          float x2 = __uint_as_float(v[4 * g + 2]) + bb.z;
          float x3 = __uint_as_float(v[4 * g + 3]) + bb.w;
          if (extras) {  // warp-uniform: PLDA row term / per-utterance bias (ECAPA attention)
            float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
            if (ub && n0 + pc + 4 * g < p.Cout) u = __ldg(reinterpret_cast<const float4*>(ub + ch * 32) + g);
            x0 += rbias + u.x; x1 += rbias + u.y; x2 += rbias + u.z; x3 += rbias + u.w;
          }
          x0 = fmaf(fmaxf(x0, relu_floor), ss.x, tt.x);
          x1 = fmaf(fmaxf(x1, relu_floor), ss.y, tt.y);
          x2 = fmaf(fmaxf(x2, relu_floor), ss.z, tt.z);
          x3 = fmaf(fmaxf(x3, relu_floor), ss.w, tt.w);
          if (extras) {
            if (act_tanh) { x0 = tanhf(x0); x1 = tanhf(x1); x2 = tanhf(x2); x3 = tanhf(x3); }
            if (act_sigmoid) {
              x0 = 1.f / (1.f + expf(-x0)); x1 = 1.f / (1.f + expf(-x1));
              x2 = 1.f / (1.f + expf(-x2)); x3 = 1.f / (1.f + expf(-x3));
            }
          }
          f[4 * g + 0] = x0; f[4 * g + 1] = x1; f[4 * g + 2] = x2; f[4 * g + 3] = x3;
        }
        if constexpr (kMask) {
          if (masked) {
#pragma unroll
            for (int j = 0; j < 16; ++j) f[j] = 0.f;
          }
        }
        if (n_tail) {
#pragma unroll
          for (int j = 0; j < 16; ++j) f[j] = n0 + pc + j < p.Cout ? f[j] : 0.f;
        }
        const int n = n0 + ch * 32;
        if (p.store_mode == 2) {
          // XVB_GEMM_STORE=reg (experiment): straight from registers, a thread owns 16 consecutive columns of its
          // row = one 32-byte sector per bf16 plane.  No slab, no barriers, no wait for the TMA engine -- but the
          // 32 scattered sectors per warp store cost more LSU time than all of that: measured 12-16 % slower on the
          // K <= 512 layers it was meant for (profiles/r01_gemm_experiments.md).  Kept as a knob.
          if (valid) {
            const long long grow = (long long)b * p.T + t;
            const int c16 = n + half * 16;
            if (planes) {
              __nv_bfloat16* dh = p.y_hi + grow * p.ldy + c16;
              __nv_bfloat16* dl = p.y_lo + grow * p.ldy + c16;
#pragma unroll
              for (int g = 0; g < 2; ++g) {
                uint32_t h[4], l[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  __nv_bfloat16 h0, l0, h1, l1;
                  split_bf16(f[g * 8 + 2 * k], h0, l0);
                  split_bf16(f[g * 8 + 2 * k + 1], h1, l1);
                  h[k] = pack_bf16x2(h0, h1);
                  l[k] = pack_bf16x2(l0, l1);
                }
                if (c16 + 8 * g < p.Cout) {   // Cout % 8 == 0 on this path
                  *reinterpret_cast<uint4*>(dh + 8 * g) = make_uint4(h[0], h[1], h[2], h[3]);
                  *reinterpret_cast<uint4*>(dl + 8 * g) = make_uint4(l[0], l[1], l[2], l[3]);
                }
              }
            }
            if (f32o) {
              float* df = p.y_f32 + grow * p.ldyf + c16;
#pragma unroll
              for (int g = 0; g < 4; ++g)
                if (c16 + 4 * g < p.Cout)     // Cout % 4 == 0 on this path
                  *reinterpret_cast<float4*>(df + 4 * g) = make_float4(f[4 * g], f[4 * g + 1], f[4 * g + 2], f[4 * g + 3]);
            }
          }
          return;
        }
        const bool direct = p.store_mode == 1;
        if (planes) {
          // the previous store must have finished reading the slab
          if (!direct && leader) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          asm volatile("bar.sync 1, 256;" ::: "memory");
          // two slabs of 64-byte rows (SWIZZLE_64B pattern): 16-byte chunk c of row r sits at c ^ ((r>>1)&3)
          const uint32_t sh = slab + row * 64, sl = slab + 8192 + row * 64;
          const int sw = (row >> 1) & 3;
#pragma unroll
          for (int g = 0; g < 2; ++g) {
            uint32_t h[4], l[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              __nv_bfloat16 h0, l0, h1, l1;
              split_bf16(f[g * 8 + 2 * k], h0, l0);
              split_bf16(f[g * 8 + 2 * k + 1], h1, l1);
              h[k] = pack_bf16x2(h0, h1);
              l[k] = pack_bf16x2(l0, l1);
            }
            const int c = half * 2 + g;
            st_shared_v4(sh + ((c ^ sw) << 4), h[0], h[1], h[2], h[3]);
            st_shared_v4(sl + ((c ^ sw) << 4), l[0], l[1], l[2], l[3]);
          }
          if (!direct) fence_proxy_async();
          asm volatile("bar.sync 2, 256;" ::: "memory");
          if (direct) {
            // transpose through the slab: a warp now owns 8 rows x 64 contiguous bytes per instruction
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int item = etid + 256 * k;
              const int plane = item >> 9, rr = (item & 511) >> 2, cc = item & 3;
              const int gb = b0 + (rr >> p.log2_tb), gt = t0 + (rr & (p.Tb - 1)), col = n + cc * 8;
              const uint4 w = ld_shared_u4(slab + plane * 8192 + rr * 64 + ((cc ^ ((rr >> 1) & 3)) << 4));
              if (gb < p.B && gt < p.T && col < p.Cout)
                *reinterpret_cast<uint4*>((plane ? p.y_lo : p.y_hi) + ((long long)gb * p.T + gt) * p.ldy + col) = w;
            }
          } else if (leader && !XVB_DBG(p, 4)) {
            tma_store_3d(&map_y_hi, slab_base, n, t0, b0);
            tma_store_3d(&map_y_lo, slab_base + 8192, n, t0, b0);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        }
        if (f32o) {
          if (!direct && leader) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          asm volatile("bar.sync 1, 256;" ::: "memory");
          // one slab of 128-byte rows (SWIZZLE_128B pattern): chunk c of row r sits at c ^ (r & 7)
          const uint32_t sf = slab + row * 128;
          const int sw = row & 7;
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            const int c = half * 4 + g;
            st_shared_v4(sf + ((c ^ sw) << 4), __float_as_uint(f[4 * g]), __float_as_uint(f[4 * g + 1]),
                         __float_as_uint(f[4 * g + 2]), __float_as_uint(f[4 * g + 3]));
          }
          if (!direct) fence_proxy_async();
          asm volatile("bar.sync 2, 256;" ::: "memory");
          if (direct) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int item = etid + 256 * k;
              const int rr = item >> 3, cc = item & 7;
              const int gb = b0 + (rr >> p.log2_tb), gt = t0 + (rr & (p.Tb - 1)), col = n + cc * 4;
              const float4 w = ld_shared_f4(slab + rr * 128 + ((cc ^ (rr & 7)) << 4));
              if (gb < p.B && gt < p.T && col < p.Cout)
                *reinterpret_cast<float4*>(p.y_f32 + ((long long)gb * p.T + gt) * p.ldyf + col) = w;
            }
          } else if (leader && !XVB_DBG(p, 4)) {
            tma_store_3d(&map_y_f32, slab_base, n, t0 + slice, b0);   // split-K: partial of slice s at "time" s
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        }
      };

      // trial histogram: score -> bin -> shared-memory counter of its class (same / different speaker).
      // Branch-free counting of the out-of-window scores (the vast majority in a zoomed pass); the
      // per-score validity test is only compiled in for ragged / diagonal tiles.
      const int lab_r = (hist && valid) ? __ldg(p.row_label + b) : -1;
      const bool plain_tile = n0 + kTileN <= p.Cout && !(p.hist_sym && n_blk == m_unit);
      const uint32_t row_ok = valid ? 1u : 0u;
      auto process_hist = [&](uint32_t (&v)[16], int ch, auto plain_tag) {
        constexpr bool kPlain = decltype(plain_tag)::value;
        const int pc = ch * 32 + half * 16;
        const float top = (float)(p.hist_bins - 2);
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const float4 bb = ld_shared_f4(prm + (pc + 4 * g) * 4);
          const float4 ll = ld_shared_f4(prm + (kTileN + pc + 4 * g) * 4);
          const float cb[4] = {bb.x, bb.y, bb.z, bb.w};
          const int cl[4] = {__float_as_int(ll.x), __float_as_int(ll.y), __float_as_int(ll.z), __float_as_int(ll.w)};
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            uint32_t ok = row_ok;
            if constexpr (!kPlain) {
              const int col = n0 + pc + 4 * g + k;
              ok = (valid && cl[k] != -2 && (!p.hist_sym || col > b)) ? 1u : 0u;
            }
            const float sc = __uint_as_float(v[4 * g + k]) + cb[k] + rbias;
            const float x = (sc - p.hist_lo) * p.hist_inv_w;
            const uint32_t cls = cl[k] == lab_r ? 1u : 0u;
            const uint32_t bl = x < 0.f ? ok : 0u;
            const uint32_t ab = !(x < top) ? ok : 0u;          // also catches NaN
            h_below[0] += bl & (cls ^ 1u); h_below[1] += bl & cls;
            h_above[0] += ab & (cls ^ 1u); h_above[1] += ab & cls;
            if (ok & ~(bl | ab))
              asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(hslab + ((int)cls * p.hist_bins + 1 + (int)x) * 4), "r"(1u) : "memory");
          }
        }
      };
      auto process_hist_any = [&](uint32_t (&v)[16], int ch) {
        if (plain_tile) process_hist(v, ch, std::true_type{});
        else process_hist(v, ch, std::false_type{});
      };

      if (!hist && p.plane_box64) {
        // Plane-only outputs (every frame layer but the last): 64-column chunks, the hi plane and then the lo plane
        // of the chunk through the 16 KB slab (128 rows x 128 bytes, SWIZZLE_128B).  Same number of barriers and slab
        // hand-overs per column as the 32-column path, but every store row is a whole 128-byte line instead of two
        // 64-byte halves written at different times: half as many write requests next to the operand stream
        // (profiles/r01_gemm_experiments.md: shorter rows cost 12-16 % on the K <= 512 layers).
        const int nch64 = XVB_DBG(p, 1) ? 0 : (min(p.Cout - n0, kTileN) + 63) >> 6;
        const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16) + acc * kTileN + half * 32;
        uint32_t v0[16], v1[16];
        tmem_ld_32x16(tq, v0);
        tmem_ld_32x16(tq + 16, v1);
#pragma unroll 1
        for (int c64 = 0; c64 < nch64; ++c64) {
          tmem_ld_wait();
          const int pc = c64 * 64 + half * 32;
          uint32_t hh[16], ll[16];
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            float4 bb = make_float4(0.1f, 0.1f, 0.1f, 0.1f), ss = make_float4(1.1f, 1.1f, 1.1f, 1.1f), tt = bb;
            if (!XVB_DBG(p, 16)) {
              bb = ld_shared_f4(prm + (pc + 4 * g) * 4);
              ss = ld_shared_f4(prm + (kTileN + pc + 4 * g) * 4);
              tt = ld_shared_f4(prm + (2 * kTileN + pc + 4 * g) * 4);
            }
            const uint32_t* src = g < 4 ? v0 + 4 * g : v1 + 4 * (g - 4);
            float x0 = __uint_as_float(src[0]) + bb.x, x1 = __uint_as_float(src[1]) + bb.y;
            float x2 = __uint_as_float(src[2]) + bb.z, x3 = __uint_as_float(src[3]) + bb.w;
            if (extras) {
              float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
              if (p.utt_bias && valid && n0 + pc + 4 * g < p.Cout)
                u = __ldg(reinterpret_cast<const float4*>(p.utt_bias + (long long)b * p.ld_utt + n0 + pc + 4 * g));
              x0 += rbias + u.x; x1 += rbias + u.y; x2 += rbias + u.z; x3 += rbias + u.w;
            }
            x0 = fmaf(fmaxf(x0, relu_floor), ss.x, tt.x);
            x1 = fmaf(fmaxf(x1, relu_floor), ss.y, tt.y);
            x2 = fmaf(fmaxf(x2, relu_floor), ss.z, tt.z);
            x3 = fmaf(fmaxf(x3, relu_floor), ss.w, tt.w);
            if (extras) {
              if (act_tanh) { x0 = tanhf(x0); x1 = tanhf(x1); x2 = tanhf(x2); x3 = tanhf(x3); }
              if (act_sigmoid) {
                x0 = 1.f / (1.f + expf(-x0)); x1 = 1.f / (1.f + expf(-x1));
                x2 = 1.f / (1.f + expf(-x2)); x3 = 1.f / (1.f + expf(-x3));
              }
            }
            if constexpr (kMask) {
              if (masked) { x0 = 0.f; x1 = 0.f; x2 = 0.f; x3 = 0.f; }
            }
            if (n_tail) {
              const int c = n0 + pc + 4 * g;
              x0 = c < p.Cout ? x0 : 0.f; x1 = c + 1 < p.Cout ? x1 : 0.f;
              x2 = c + 2 < p.Cout ? x2 : 0.f; x3 = c + 3 < p.Cout ? x3 : 0.f;
            }
            __nv_bfloat16 h0, l0, h1, l1, h2, l2, h3, l3;
            split_bf16(x0, h0, l0); split_bf16(x1, h1, l1); split_bf16(x2, h2, l2); split_bf16(x3, h3, l3);
            hh[2 * g] = pack_bf16x2(h0, h1); hh[2 * g + 1] = pack_bf16x2(h2, h3);
            ll[2 * g] = pack_bf16x2(l0, l1); ll[2 * g + 1] = pack_bf16x2(l2, l3);
          }
          if (c64 + 1 < nch64) {                             // the accumulator values are consumed: fetch the next chunk
            tmem_ld_32x16(tq + (c64 + 1) * 64, v0);
            tmem_ld_32x16(tq + (c64 + 1) * 64 + 16, v1);
          }
          const int ncol = n0 + c64 * 64;
          const uint32_t rowaddr = slab + row * 128;
          const int sw = row & 7;
#pragma unroll
          for (int plane = 0; plane < 2; ++plane) {
            if (p.store_mode == 1) {
              // XVB_GEMM_STORE=direct (experiment): the slab is drained by the epilogue threads themselves -- 16 bytes per
              // thread, a warp instruction covers four whole 128-byte lines -- instead of by the TMA unit
              asm volatile("bar.sync 1, 256;" ::: "memory");          // everybody has read the previous contents
              const uint32_t* wd = plane == 0 ? hh : ll;
#pragma unroll
              for (int k = 0; k < 4; ++k)
                st_shared_v4(rowaddr + (((half * 4 + k) ^ sw) << 4), wd[4 * k], wd[4 * k + 1], wd[4 * k + 2], wd[4 * k + 3]);
              asm volatile("bar.sync 2, 256;" ::: "memory");
              __nv_bfloat16* base = plane == 0 ? p.y_hi : p.y_lo;
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const int item = etid + 256 * k;
                const int rr = item >> 3, cc = item & 7;
                const int gb = b0 + (rr >> p.log2_tb), gt = t0 + (rr & (p.Tb - 1)), col = ncol + cc * 8;
                const uint4 wv = ld_shared_u4(slab + rr * 128 + ((cc ^ (rr & 7)) << 4));
                if (gb < p.B && gt < p.T && col < p.Cout)
                  *reinterpret_cast<uint4*>(base + ((long long)gb * p.T + gt) * p.ldy + col) = wv;
              }
              continue;
            }
            if (leader) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            if (!XVB_DBG(p, 64)) asm volatile("bar.sync 1, 256;" ::: "memory");
            const uint32_t* w = plane == 0 ? hh : ll;
            if (!XVB_DBG(p, 32)) {
#pragma unroll
              for (int k = 0; k < 4; ++k)                      // this thread's 32 columns = 4 chunks of 16 bytes
                st_shared_v4(rowaddr + (((half * 4 + k) ^ sw) << 4), w[4 * k], w[4 * k + 1], w[4 * k + 2], w[4 * k + 3]);
            } else if (w[0] == 0x12345678u) {                  // keep the values live
              st_shared_v4(rowaddr, w[0], w[5], w[10], w[15]);
            }
            fence_proxy_async();
            if (!XVB_DBG(p, 64)) asm volatile("bar.sync 2, 256;" ::: "memory");
            if (leader && !XVB_DBG(p, 4)) {
              tma_store_3d(plane == 0 ? &map_y_hi : &map_y_lo, slab_base, ncol, t0, b0);
              asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
          }
        }
        tcgen05_fence_before();
        if constexpr (kCta == 1) mbar_arrive(&tmem_empty_bar[acc]);
        else mbar_arrive_cluster(&tmem_empty_bar[acc], 0);
        continue;
      }
      uint32_t va[16], vb[16];
      int ch = 0;
      if (XVB_DBG(p, 1)) ch = nch;
      else tmem_ld_32x16(trow, va);
      while (ch < nch) {
        tmem_ld_wait();
        if (ch + 1 < nch && !XVB_DBG(p, 8)) tmem_ld_32x16(trow + (ch + 1) * 32, vb);
        if constexpr (hist) process_hist_any(va, ch); else process(va, ch);
        if (++ch >= nch) break;
        tmem_ld_wait();
        if (ch + 1 < nch && !XVB_DBG(p, 8)) tmem_ld_32x16(trow + (ch + 1) * 32, va);
        if constexpr (hist) process_hist_any(vb, ch); else process(vb, ch);
        ++ch;
      }
      tcgen05_fence_before();
      if constexpr (kCta == 1) mbar_arrive(&tmem_empty_bar[acc]);
      else mbar_arrive_cluster(&tmem_empty_bar[acc], 0);  // the leader's barrier counts both CTAs' epilogues
      if (hist && (it & 0x3fffu) == 0) hist_flush();      // u32 counters: <= 2^14 tiles x 2^15 scores between flushes
    }
    if (hist) hist_flush();
    if (leader) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // stores complete before exit
  }

  tcgen05_fence_before();
  __syncthreads();
  if constexpr (kCta == 2) cluster_sync();  // nobody leaves while the pair still reads its smem / barriers
  if (warp == 1) tmem_dealloc<kCta>(tmem_base, Cfg::kTmemCols);
}

// Split-K tail: y[b,c] = epi(sum_s part[b,s,c]) with the slices added in index order (deterministic),
// same epilogue order as the GEMM's: +bias -> ReLU -> BN -> tanh/sigmoid -> fp32 and/or split planes.
__global__ void segment_reduce_kernel(const float* __restrict__ part, int S, int B, int Cout, const float* __restrict__ bias,
                                      const float* __restrict__ scale, const float* __restrict__ shift, int flags,
                                      float* __restrict__ y_f32, long long ldyf, __nv_bfloat16* __restrict__ y_hi,
                                      __nv_bfloat16* __restrict__ y_lo, long long ldy) {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (idx >= (long long)B * Cout) return;
  const int b = (int)(idx / Cout), c = (int)(idx - (long long)b * Cout);
  const float* src = part + (long long)b * S * Cout + c;
  float x = src[0];
  for (int s = 1; s < S; ++s) x += src[(long long)s * Cout];
  x += bias ? bias[c] : 0.f;
  if (flags & XVB_RELU) x = fmaxf(x, 0.f);
  if (flags & XVB_BN) x = fmaf(x, scale[c], shift[c]);
  if (flags & XVB_TANH) x = tanhf(x);
  if (flags & XVB_SIGMOID) x = 1.f / (1.f + expf(-x));
  if (y_f32) y_f32[(long long)b * ldyf + c] = x;
  if (y_hi) {
    __nv_bfloat16 h, l;
    split_bf16(x, h, l);
    y_hi[(long long)b * ldy + c] = h;
    y_lo[(long long)b * ldy + c] = l;
  }
}

// ------------------------------------------------------------------------------------------------
// Host side: tensor maps + launch
// ------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  });
  return fn;
}

// Generic tiled tensor map (exported for pooling.cu).  esize 2 -> bf16, 4 -> fp32; swizzle_bytes 0/64/128.
int make_tensor_map(CUtensorMap* m, const void* base, int esize, int rank, const unsigned long long* dims,
                    const unsigned long long* strides_bytes, const unsigned* box, int swizzle_bytes) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point not available"); return XVB_ECUDA; }
  cuuint64_t d[5], st[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) { d[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
  for (int i = 0; i + 1 < rank; ++i) st[i] = strides_bytes[i];
  const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                               : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = enc(m, esize == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, rank,
                   const_cast<void*>(base), d, st, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(rank %d) failed: %d", rank, (int)r); return XVB_ECUDA; }
  return XVB_OK;
}

// (C, T, B) bf16 frame matrix with row pitch ld; box = 64 channels x Tb frames x Bb utterances.
static int make_frame_map(CUtensorMap* m, const void* base, int C, int T, int B, long long ld, int Tb, int Bb,
                          long long batch_stride = 0) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point not available"); return XVB_ECUDA; }
  cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)T, (cuuint64_t)B};
  cuuint64_t strides[2] = {(cuuint64_t)ld * 2, batch_stride ? (cuuint64_t)batch_stride * 2 : (cuuint64_t)ld * 2 * (cuuint64_t)T};
  cuuint32_t box[3] = {(cuuint32_t)kBlockK, (cuuint32_t)Tb, (cuuint32_t)Bb};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(frame map C=%d T=%d B=%d ld=%lld) failed: %d", C, T, B, ld, (int)r); return XVB_ECUDA; }
  return XVB_OK;
}

// (K, Cout) bf16 packed weight, K contiguous; box = 64 x block_n.
static int make_weight_map(CUtensorMap* m, const void* base, long long K, int Cout, int block_n) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point not available"); return XVB_ECUDA; }
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)Cout};
  cuuint64_t strides[1] = {(cuuint64_t)K * 2};
  cuuint32_t box[2] = {(cuuint32_t)kBlockK, (cuuint32_t)block_n};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(weight map K=%lld Cout=%d) failed: %d", K, Cout, (int)r); return XVB_ECUDA; }
  return XVB_OK;
}

// XVB_GEMM_CTA=1 forces single-CTA tiles, =2 (default) uses CTA pairs for the big layers.
static int gemm_cta_mode() {
  static int mode = 0;
  if (mode == 0) {
    const char* e = getenv("XVB_GEMM_CTA");
    mode = (e && e[0] == '1') ? 1 : 2;
  }
  return mode;
}

// Epilogue store path: TMA stores from the swizzled slab (default), or XVB_GEMM_STORE=direct for
// coalesced st.global after a transpose through the same slab (measured 5-10 % slower, kept as a knob).
static int gemm_store_mode() {   // -1: automatic (per layer shape)
  static int mode = -2;
  if (mode == -2) {
    const char* e = getenv("XVB_GEMM_STORE");
    mode = !e ? -1 : e[0] == 'd' ? 1 : e[0] == 'r' ? 2 : e[0] == 't' ? 0 : -1;
  }
  return mode;
}

// Pick the (Tb, Bb) factorisation of the 128-row M tile with the fewest padded rows.
static void choose_m_tile(int B, int T, int* Tb_out, int* Bb_out, int max_tb = 128) {
  if (T == 1) {   // segment-level layers: one row per utterance.  (Also what split-K's "slice as time" store
    *Tb_out = 1;  // relies on: a box taller than one frame would spill zeros into the next slices' rows.)
    *Bb_out = 128;
    return;
  }
  long long best = -1;
  int bt = max_tb;
  for (int Tb = max_tb; Tb >= 1; Tb >>= 1) {
    const int Bb = 128 / Tb;
    const long long rows = (long long)((T + Tb - 1) / Tb) * Tb * ((B + Bb - 1) / Bb) * Bb;
    if (best < 0 || rows < best) { best = rows; bt = Tb; }
  }
  *Tb_out = bt;
  *Bb_out = 128 / bt;
}

// Output tensor map: (Cout, T, B) with row pitch ld elements of `esize` bytes; box = 32 columns x
// Tb x Bb; 64-byte rows (bf16) use SWIZZLE_64B, 128-byte rows (fp32) SWIZZLE_128B.
static int make_out_map(CUtensorMap* m, const void* base, int esize, int C, int T, int B, long long ld, int Tb, int Bb,
                        int box_cols = 32) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point not available"); return XVB_ECUDA; }
  cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)T, (cuuint64_t)B};
  cuuint64_t strides[2] = {(cuuint64_t)ld * esize, (cuuint64_t)ld * esize * (cuuint64_t)T};
  cuuint32_t box[3] = {(cuuint32_t)box_cols, (cuuint32_t)Tb, (cuuint32_t)Bb};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(m, esize == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3,
                   const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   box_cols * esize == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(output map C=%d T=%d B=%d ld=%lld) failed: %d", C, T, B, ld, (int)r); return XVB_ECUDA; }
  return XVB_OK;
}

// ------------------------------------------------------------------------------------------------
// Plan / launch split.  Everything that depends only on shapes and pointers -- tile geometry, the nine
// tensor maps (cuTensorMapEncodeTiled is a ~1 us driver call each), the kernel instantiation, the grid --
// is decided once in a GemmPlan; launching a plan is one cudaLaunchKernelEx (+ the split-K reduce).  The
// extractor objects keep their plans per (B, T), so a batch costs launches only (C1 latency, VERDICT r1 #9).
// ------------------------------------------------------------------------------------------------
struct GemmPlan {
  CUtensorMap ma_hi, ma_lo, ma2_hi, ma2_lo, mw_hi, mw_lo, my_hi, my_lo, my_f32;
  TdnnGemmParams p;
  int (*launch)(const GemmPlan&, const CUtensorMap&, cudaStream_t) = nullptr;   // nullptr: this shard owns no rows
  int grid = 0;
  int pdl = 1;
  // split-K tail (segment_reduce_kernel); the GEMM itself then writes fp32 partials into `scratch`
  bool reduce = false;
  const float* r_bias = nullptr; const float* r_scale = nullptr; const float* r_shift = nullptr;
  int r_flags = 0;
  float* r_y_f32 = nullptr; long long r_ldyf = 0;
  __nv_bfloat16* r_y_hi = nullptr; __nv_bfloat16* r_y_lo = nullptr; long long r_ldy = 0;
  int out_Tdim = 0;          // time extent of the fp32 output map (k_slices for split-K)
};

template <int BLOCK_N, int kCta, int kNSub, bool kPool, bool kHist, bool kMask>
static int launch_inst(const GemmPlan& pl, const CUtensorMap& my_f32, cudaStream_t stream) {
  using Cfg = GemmCfg<BLOCK_N, kCta, kNSub>;
  XVB_ENSURE_DYN_SMEM((tdnn_gemm_bf16x3_kernel<BLOCK_N, kCta, kNSub, kPool, kHist, kMask>), Cfg::kSmemBytes);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(pl.grid);
  cfg.blockDim = dim3(kNumThreads);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kCta;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pl.pdl ? 2 : 1;
  XVB_CUDA(cudaLaunchKernelEx(&cfg, tdnn_gemm_bf16x3_kernel<BLOCK_N, kCta, kNSub, kPool, kHist, kMask>, pl.ma_hi, pl.ma_lo, pl.ma2_hi,
                              pl.ma2_lo, pl.mw_hi, pl.mw_lo, pl.my_hi, pl.my_lo, my_f32, pl.p));
  XVB_LAUNCH_CHECK();
  return XVB_OK;
}

template <int BLOCK_N, int kCta, int kNSub = 1, bool kPool = false, bool kHist = false, bool kMask = false>
static int prepare_gemm(GemmPlan& pl, const void* w_hi, const void* w_lo) {
  using Cfg = GemmCfg<BLOCK_N, kCta, kNSub>;
  TdnnGemmParams& p = pl.p;
  const long long K = (long long)p.ntaps * p.cin_p16;
  int rc = make_weight_map(&pl.mw_hi, w_hi, K, p.Cout, Cfg::kBRows);
  if (rc) return rc;
  rc = make_weight_map(&pl.mw_lo, w_lo, K, p.Cout, Cfg::kBRows);
  if (rc) return rc;
  p.num_n_blk = (p.Cout + Cfg::kTileN - 1) / Cfg::kTileN;
  const int all_m_units = (p.num_t_blk * p.num_b_blk + kCta - 1) / kCta;  // 128-row blocks, or pairs of them
  if (p.unit_first >= all_m_units) { pl.launch = nullptr; return XVB_OK; }  // this shard owns no rows
  const int num_m_units = (all_m_units - p.unit_first + p.unit_stride - 1) / p.unit_stride;
  p.num_units = num_m_units;
  p.hist_group = 8;
  const long long tiles = kHist ? (long long)((num_m_units + p.hist_group - 1) / p.hist_group) * p.hist_group * p.num_n_blk
                                : (long long)num_m_units * p.num_n_blk * (p.k_slices > 1 ? p.k_slices : 1);
  XVB_CHECK_ARG(tiles < (1ll << 31), "xvb_tdnn_affine: %d x %d tiles exceed one launch", num_m_units, p.num_n_blk);
  p.num_tiles = (int)tiles;
#ifdef XVB_TIMING_EXPERIMENTS
  p.debug = getenv("XVB_GEMM_DEBUG") ? atoi(getenv("XVB_GEMM_DEBUG")) : 0;
#endif
  static const int box64_knob = getenv("XVB_GEMM_BOX64") ? atoi(getenv("XVB_GEMM_BOX64")) : 1;
  p.plane_box64 = (box64_knob && !kPool && !kHist && p.y_hi && !p.y_f32 && p.store_mode <= 1 && Cfg::kTileN >= 64) ? 1 : 0;
  if (p.y_hi) {
    const int bc = p.plane_box64 ? 64 : 32;
    if ((rc = make_out_map(&pl.my_hi, p.y_hi, 2, p.Cout, p.T, p.B, p.ldy, p.Tb, p.Bb, bc))) return rc;
    if ((rc = make_out_map(&pl.my_lo, p.y_lo, 2, p.Cout, p.T, p.B, p.ldy, p.Tb, p.Bb, bc))) return rc;
  } else {
    pl.my_hi = pl.mw_hi; pl.my_lo = pl.mw_lo;  // unused
  }
  pl.out_Tdim = p.k_slices > 1 ? p.k_slices : p.T;
  if (p.y_f32) {
    if ((rc = make_out_map(&pl.my_f32, p.y_f32, 4, p.Cout, pl.out_Tdim, p.B, p.ldyf, p.Tb, p.Bb))) return rc;
  } else {
    pl.my_f32 = pl.mw_hi;  // unused
  }
  const int units = sm_count() / kCta;  // CTAs (kCta=1) or CTA pairs (kCta=2) resident at once
  pl.grid = (p.num_tiles < units ? p.num_tiles : units) * kCta;
  static const int pdl = getenv("XVB_PDL") ? atoi(getenv("XVB_PDL")) : 1;
  pl.pdl = pdl;
  pl.launch = &launch_inst<BLOCK_N, kCta, kNSub, kPool, kHist, kMask>;
  return XVB_OK;
}

// Split-K for segment-level layers (T == 1: M = B rows, tdnn6 has K = 3000): the slice count depends
// on K only, so a sub-batch reproduces the full batch's rows bit for bit.  Returns the number of slices (1 = off).
static int splitk_slices(const xvb_tdnn_args_t& a, bool has_hist, int* kb_per_slice) {
  const int num_cblk = (a.Cin + kBlockK - 1) / kBlockK;
  *kb_per_slice = num_cblk;
  const int splitk = getenv("XVB_SPLITK") ? atoi(getenv("XVB_SPLITK")) : 1;   // read per plan: tests flip it
  if (!(splitk && a.T == 1 && a.ntaps == 1 && !a.x2_hi && !a.pool_partial && !has_hist && !a.row_bias && !a.utt_bias &&
        a.B <= 1024 && num_cblk >= 24 && a.Cout % 4 == 0))
    return 1;
  int S = num_cblk / 6;
  S = S > 8 ? 8 : S;
  *kb_per_slice = (num_cblk + S - 1) / S;
  return (num_cblk + *kb_per_slice - 1) / *kb_per_slice;   // every slice owns >= 1 channel block
}

}  // namespace xvb

using namespace xvb;

size_t xvb::gemm_plan_scratch_bytes(const xvb_tdnn_args_t& a, const TrialHist* th) {
  int kb;
  const int S = splitk_slices(a, th != nullptr, &kb);
  return S > 1 ? (size_t)a.B * S * a.Cout * sizeof(float) : 0;
}

int xvb::gemm_plan_build(GemmPlan** out, const xvb_tdnn_args_t& a, const TrialHist* th, void* scratch) {
  int rc = require_sm100();
  if (rc) return rc;
  *out = nullptr;
  const int B = a.B, T = a.T, Cin = a.Cin, Cout = a.Cout, ntaps = a.ntaps;
  XVB_CHECK_ARG(a.x_hi && a.x_lo && a.w_hi && a.w_lo, "xvb_tdnn_affine: null operand pointer");
  XVB_CHECK_ARG(B > 0 && T > 0 && Cin > 0 && Cout > 0, "xvb_tdnn_affine: bad shape B=%d T=%d Cin=%d Cout=%d", B, T, Cin, Cout);
  XVB_CHECK_ARG(ntaps >= 1 && ntaps <= XVB_MAX_TAPS && a.context_host, "xvb_tdnn_affine: ntaps=%d out of range", ntaps);
  if (a.x_batch_stride)   // im2col view: overlapping rows
    XVB_CHECK_ARG(a.ldx % 8 == 0 && a.x_batch_stride % 8 == 0 && !a.x2_hi && ntaps == 1 &&
                  a.x_batch_stride >= (long long)(T - 1) * a.ldx + Cin,
                  "xvb_tdnn_affine: x_batch_stride=%lld needs ntaps==1, no second source, 8-element alignment and room for T windows",
                  (long long)a.x_batch_stride);
  else
    XVB_CHECK_ARG(a.ldx % 8 == 0 && a.ldx >= Cin, "xvb_tdnn_affine: ldx=%lld must be a multiple of 8 and >= Cin", (long long)a.ldx);
  XVB_CHECK_ARG((a.x2_hi != nullptr) == (a.x2_lo != nullptr), "xvb_tdnn_affine: x2_hi/x2_lo must both be set or both NULL");
  if (a.x2_hi) XVB_CHECK_ARG(a.ldx2 % 8 == 0 && a.ldx2 >= Cin, "xvb_tdnn_affine: ldx2=%lld must be a multiple of 8 and >= Cin", (long long)a.ldx2);
  XVB_CHECK_ARG((a.y_hi != nullptr) == (a.y_lo != nullptr), "xvb_tdnn_affine: y_hi/y_lo must both be set or both NULL");
  XVB_CHECK_ARG(a.y_hi || a.y_f32 || a.pool_partial || th, "xvb_tdnn_affine: no output requested");
  if (a.pool_partial) XVB_CHECK_ARG(!a.y_hi && !a.y_f32 && Cout % 4 == 0 && (uintptr_t)a.pool_partial % 16 == 0,
                                    "xvb_tdnn_affine: pool_partial excludes other outputs and needs Cout%%4==0");
  if (a.y_hi) XVB_CHECK_ARG(a.ldy % 8 == 0 && a.ldy >= Cout, "xvb_tdnn_affine: plane output needs ldy%%8==0 and ldy>=Cout");
  if (a.y_f32) XVB_CHECK_ARG(a.ldyf % 4 == 0 && a.ldyf >= Cout, "xvb_tdnn_affine: fp32 output needs ldyf%%4==0 and ldyf>=Cout");
  XVB_CHECK_ARG(!(a.flags & XVB_BN) || (a.bn_scale && a.bn_shift), "xvb_tdnn_affine: XVB_BN without scale/shift");
  if (a.utt_bias) XVB_CHECK_ARG(a.ld_utt_bias % 4 == 0 && a.ld_utt_bias >= Cout && Cout % 4 == 0 && (uintptr_t)a.utt_bias % 16 == 0,
                                "xvb_tdnn_affine: utt_bias needs ld%%4==0, Cout%%4==0, 16-byte alignment");
  XVB_CHECK_ARG(((uintptr_t)a.x_hi | (uintptr_t)a.x_lo | (uintptr_t)a.x2_hi | (uintptr_t)a.x2_lo | (uintptr_t)a.w_hi |
                 (uintptr_t)a.w_lo | (uintptr_t)a.y_hi | (uintptr_t)a.y_lo | (uintptr_t)a.y_f32) % 16 == 0,
                "xvb_tdnn_affine: pointers must be 16-byte aligned");
  for (int i = 1; i < ntaps; ++i)
    XVB_CHECK_ARG(a.context_host[i] > a.context_host[i - 1], "xvb_tdnn_affine: context must be strictly increasing (components.py:34-36)");

  GemmPlan* plp = new GemmPlan();
  struct Guard { GemmPlan* p; ~Guard() { delete p; } } guard{plp};
  GemmPlan& pl = *plp;
  TdnnGemmParams& p = pl.p;
  p = TdnnGemmParams{};
  p.B = B; p.T = T; p.Cin = Cin; p.Cout = Cout;
  choose_m_tile(B, T, &p.Tb, &p.Bb);
  p.num_t_blk = (T + p.Tb - 1) / p.Tb;
  p.num_b_blk = (B + p.Bb - 1) / p.Bb;
  p.ntaps = ntaps;
  p.cin_p16 = (int)round_up(Cin, 16);
  p.num_cblk = (Cin + kBlockK - 1) / kBlockK;
  for (int i = 0; i < ntaps; ++i) p.ctx[i] = a.context_host[i];
  p.flags = a.flags;
  p.bias = a.bias; p.scale = a.bn_scale; p.shift = a.bn_shift; p.row_bias = a.row_bias;
  p.utt_bias = a.utt_bias; p.ld_utt = a.ld_utt_bias;
  p.pool_partial = a.pool_partial;
  p.num_src = a.x2_hi ? 2 : 1;
  p.unit_first = 0; p.unit_stride = 1;
  if (th) {
    p.hist = th->hist; p.row_label = th->row_label; p.col_label = th->col_label;
    p.hist_lo = th->lo; p.hist_inv_w = th->inv_w; p.hist_bins = th->nbins; p.hist_sym = th->symmetric;
    p.unit_first = th->unit_first; p.unit_stride = th->unit_stride;
  }
  p.log2_tb = 0;
  while ((1 << p.log2_tb) < p.Tb) ++p.log2_tb;
  p.store_mode = gemm_store_mode();
  if (p.store_mode < 0) p.store_mode = 0;   // TMA stores; `reg` / `direct` measured slower (profiles/r01_gemm_experiments.md)
  if (p.store_mode >= 1) {  // vector stores need whole 16-byte groups inside the row
    if (a.y_hi) XVB_CHECK_ARG(Cout % 8 == 0, "xvb_tdnn_affine: plane output needs Cout%%8==0 (Cout=%d)", Cout);
    if (a.y_f32) XVB_CHECK_ARG(Cout % 4 == 0, "xvb_tdnn_affine: fp32 output needs Cout%%4==0 (Cout=%d)", Cout);
  }
  p.y_hi = reinterpret_cast<__nv_bfloat16*>(a.y_hi);
  p.y_lo = reinterpret_cast<__nv_bfloat16*>(a.y_lo);
  p.ldy = a.ldy; p.y_f32 = a.y_f32; p.ldyf = a.ldyf;
  p.lengths = th ? nullptr : a.lengths;   // the histogram mode has no frames

  p.k_slices = splitk_slices(a, th != nullptr, &p.kb_per_slice);
  if (p.k_slices > 1) {
    XVB_CHECK_ARG(scratch, "xvb_tdnn_affine: split-K plan needs %zu bytes of scratch", gemm_plan_scratch_bytes(a, th));
    pl.reduce = true;
    pl.r_bias = a.bias; pl.r_scale = a.bn_scale; pl.r_shift = a.bn_shift; pl.r_flags = a.flags;
    pl.r_y_f32 = a.y_f32; pl.r_ldyf = a.ldyf;
    pl.r_y_hi = reinterpret_cast<__nv_bfloat16*>(a.y_hi); pl.r_y_lo = reinterpret_cast<__nv_bfloat16*>(a.y_lo); pl.r_ldy = a.ldy;
    p.y_hi = nullptr; p.y_lo = nullptr;
    p.y_f32 = static_cast<float*>(scratch); p.ldyf = Cout;
    p.bias = nullptr; p.scale = nullptr; p.shift = nullptr; p.flags = 0;
    p.store_mode = 0;
    p.lengths = nullptr;   // segment level: one row per utterance, nothing to mask
  }

  if ((rc = make_frame_map(&pl.ma_hi, a.x_hi, Cin, T, B, a.ldx, p.Tb, p.Bb, a.x_batch_stride))) return rc;
  if ((rc = make_frame_map(&pl.ma_lo, a.x_lo, Cin, T, B, a.ldx, p.Tb, p.Bb, a.x_batch_stride))) return rc;
  if (a.x2_hi) {
    if ((rc = make_frame_map(&pl.ma2_hi, a.x2_hi, Cin, T, B, a.ldx2, p.Tb, p.Bb))) return rc;
    if ((rc = make_frame_map(&pl.ma2_lo, a.x2_lo, Cin, T, B, a.ldx2, p.Tb, p.Bb))) return rc;
  } else {
    pl.ma2_hi = pl.ma_hi; pl.ma2_lo = pl.ma_lo;  // unused
  }

  // Wide N tiles (CTA pairs) when there are enough M tiles to fill the machine, narrow ones for
  // the segment-level layers (M = B rows) so that more SMs get a tile.
  const long long m_tiles = (long long)p.num_t_blk * p.num_b_blk * p.k_slices;   // independent work items along M (and K slices)
  const int sms = sm_count();
  const int mode = gemm_cta_mode();
  const void* w_hi = a.w_hi;
  const void* w_lo = a.w_lo;
  auto dispatch = [&](auto mask_tag) -> int {
    constexpr bool kM = decltype(mask_tag)::value;
    if (a.pool_partial)  // fused pooling always runs on the swapped CTA-pair kernel (any shape: TMA zero-fills)
      return prepare_gemm<256, 2, 1, true, false, kM>(pl, w_hi, w_lo);
    if (th)              // the diagonal test of the symmetric mode assumes 256-row units x 256-column tiles
      return prepare_gemm<256, 2, 1, false, true>(pl, w_hi, w_lo);
    static const int force_bn = getenv("XVB_GEMM_BN") ? atoi(getenv("XVB_GEMM_BN")) : 0;  // tuning knobs
    // wide tiles cut the operand stream by 25-37 % but serialise the epilogue with the MMAs (one
    // accumulator in TMEM); measured slower end to end (profiles/r01_gemm_experiments.md), so opt-in.
    static const int wide = getenv("XVB_GEMM_WIDE") ? atoi(getenv("XVB_GEMM_WIDE")) : 0;
    if (mode == 2 && wide && force_bn != 128 && Cout >= 512 && (m_tiles / 2) * ((Cout + 511) / 512) >= sms / 2)
      return prepare_gemm<256, 2, 2, false, false, kM>(pl, w_hi, w_lo);
    if (mode == 2 && force_bn != 128 && Cout >= 256 && m_tiles * ((Cout + 255) / 256) >= sms)
      return prepare_gemm<256, 2, 1, false, false, kM>(pl, w_hi, w_lo);
    if (mode == 2 && Cout >= 128 && m_tiles * ((Cout + 127) / 128) >= sms)
      return prepare_gemm<128, 2, 1, false, false, kM>(pl, w_hi, w_lo);
    if (Cout >= 256 && m_tiles * ((Cout + 255) / 256) >= sms) return prepare_gemm<256, 1, 1, false, false, kM>(pl, w_hi, w_lo);
    if (Cout >= 128 && m_tiles * ((Cout + 127) / 128) >= sms) return prepare_gemm<128, 1, 1, false, false, kM>(pl, w_hi, w_lo);
    if (Cout >= 64 && m_tiles * ((Cout + 63) / 64) >= sms / 2) return prepare_gemm<64, 1, 1, false, false, kM>(pl, w_hi, w_lo);
    return prepare_gemm<32, 1, 1, false, false, kM>(pl, w_hi, w_lo);
  };
  if ((rc = p.lengths ? dispatch(std::true_type{}) : dispatch(std::false_type{}))) return rc;
  guard.p = nullptr;
  *out = plp;
  return XVB_OK;
}

void xvb::gemm_plan_destroy(GemmPlan* pl) { delete pl; }

// Launch a plan.  `y_f32_override` (optional) redirects the fp32 output of this launch to another buffer of the
// same shape and pitch (the extractors' last layer writes straight into the caller's embedding matrix): for a
// split-K plan it is just the reduce kernel's pointer, otherwise the one output tensor map is re-encoded.
int xvb::gemm_plan_launch(const GemmPlan* plp, void* stream, float* y_f32_override) {
  const GemmPlan& pl = *plp;
  if (!pl.launch) return XVB_OK;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  int rc;
  if (!pl.reduce && y_f32_override && y_f32_override != pl.p.y_f32) {
    XVB_CHECK_ARG(pl.p.y_f32 && !pl.p.hist && !pl.p.pool_partial && (uintptr_t)y_f32_override % 16 == 0,
                  "gemm_plan_launch: this plan has no fp32 output to redirect");
    GemmPlan tmp = pl;
    tmp.p.y_f32 = y_f32_override;
    if ((rc = make_out_map(&tmp.my_f32, y_f32_override, 4, pl.p.Cout, pl.out_Tdim, pl.p.B, pl.p.ldyf, pl.p.Tb, pl.p.Bb))) return rc;
    return tmp.launch(tmp, tmp.my_f32, s);
  }
  if ((rc = pl.launch(pl, pl.my_f32, s))) return rc;
  if (!pl.reduce) return XVB_OK;
  float* yf = y_f32_override ? y_f32_override : pl.r_y_f32;
  const long long n = (long long)pl.p.B * pl.p.Cout;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)((n + 255) / 256));
  cfg.blockDim = dim3(256);
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  XVB_CUDA(cudaLaunchKernelEx(&cfg, segment_reduce_kernel, (const float*)pl.p.y_f32, pl.p.k_slices, pl.p.B, pl.p.Cout, pl.r_bias,
                              pl.r_scale, pl.r_shift, pl.r_flags, yf, pl.r_ldyf, pl.r_y_hi, pl.r_y_lo, pl.r_ldy));
  XVB_LAUNCH_CHECK();
  return XVB_OK;
}

int xvb::tdnn_affine_impl(const xvb_tdnn_args_t& a, void* stream, const TrialHist* th) {
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  TempBuf partial(s);
  int rc;
  XVB_CHECK_ARG(a.B > 0 && a.Cin > 0 && a.Cout > 0, "xvb_tdnn_affine: bad shape B=%d Cin=%d Cout=%d", a.B, a.Cin, a.Cout);
  const size_t need = gemm_plan_scratch_bytes(a, th);
  if (need && (rc = partial.alloc(need))) return rc;
  GemmPlan* pl = nullptr;
  if ((rc = gemm_plan_build(&pl, a, th, partial.p))) return rc;
  rc = gemm_plan_launch(pl, stream, nullptr);
  gemm_plan_destroy(pl);
  return rc;
}

extern "C" int xvb_pool_partial_blocks(int B, int T, int* frames_per_block) {
  int Tb, Bb;
  choose_m_tile(B, T, &Tb, &Bb);
  if (frames_per_block) *frames_per_block = Tb;
  return (T + Tb - 1) / Tb;
}

extern "C" int xvb_tdnn_affine_ex(const xvb_tdnn_args_t* args, void* stream) {
  XVB_CHECK_ARG(args, "xvb_tdnn_affine_ex: null args");
  return tdnn_affine_impl(*args, stream);
}

extern "C" int xvb_tdnn_affine(const uint16_t* x_hi, const uint16_t* x_lo, int64_t ldx, const uint16_t* w_hi,
                               const uint16_t* w_lo, const float* bias, const float* bn_scale, const float* bn_shift,
                               int flags, const int* context_host, int ntaps, uint16_t* y_hi, uint16_t* y_lo,
                               int64_t ldy, float* y_f32, int64_t ldyf, int B, int T, int Cin, int Cout,
                               void* stream) {
  xvb_tdnn_args_t a{};
  a.x_hi = x_hi; a.x_lo = x_lo; a.ldx = ldx; a.w_hi = w_hi; a.w_lo = w_lo;
  a.bias = bias; a.bn_scale = bn_scale; a.bn_shift = bn_shift; a.flags = flags;
  a.context_host = context_host; a.ntaps = ntaps;
  a.y_hi = y_hi; a.y_lo = y_lo; a.ldy = ldy; a.y_f32 = y_f32; a.ldyf = ldyf;
  a.B = B; a.T = T; a.Cin = Cin; a.Cout = Cout;
  return tdnn_affine_impl(a, stream);
}
