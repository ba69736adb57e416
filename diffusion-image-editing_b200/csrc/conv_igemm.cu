// Implicit-GEMM convolution / linear layer on the 5th-gen tensor cores (tcgen05, sm_100a).
//
//   out[n,h,w,co] = sum_{tap, c} A[n, h*s+dh(tap), w*s+dw(tap), c] * Wt[co, tap, c]  (+ epilogue)
//
// GEMM view: M = output pixels (128 per CTA: an Nt x Ht x Wt brick of the NHWC output),
// N = output channels (BN per CTA), K = taps x input channels, walked 64 channels at a time.
//  * A is never materialised (no im2col buffer): for every (tap, 64-channel chunk) one TMA
//    tiled load fetches the shifted Nt x Ht x Wt x 64 brick of the NHWC activation straight
//    into a 128B-swizzled K-major smem tile; the conv zero padding is TMA out-of-bounds fill.
//    Stride-2 convolutions view the input as (2C, W/2, 2, H/2, N) so a tap is again a box.
//    The K loop can draw chunks from two tensors (skip concatenation without a copy).
//    After the taps, an optional 1x1 "residual segment" (K chunks read at the output pixel from up to
//    two more tensors, weights appended to B along K) fuses the ResNet shortcut convolution or, with
//    identity weights, the residual add - the epilogue never reads the residual.
//  * B (weights, f16 [Cout][tap][Cin | residual]) is a plain 2-D TMA tile.
//  * one elected thread issues tcgen05.mma (UMMA 128 x BN x 16, f16 in, fp32 accumulate in
//    TMEM); tcgen05.commit releases smem stages / signals the epilogue through mbarriers.
//  * warp roles: warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2-5 =
//    epilogue (tcgen05.ld TMEM -> registers, + bias + time-embedding, f16 tile staged in 128B-swizzled
//    smem and written with one TMA store per 64-channel slab; fp32 NCHW direct store for conv_out).  Persistent CTAs (one per SM), 6-8 stage smem ring that never drains
//    between tiles, double-buffered TMEM accumulator so the epilogue overlaps the next main loop.
#include "conv_igemm.cuh"
#include "gn_math.cuh"
#include "tcgen05_ptx.cuh"

#include <cudaTypedefs.h>
#include <stdlib.h>
#include <vector>

namespace b2e {

// TMA producer warp (non-halo kernels: the A operand) + MMA warp + 4 epilogue warps + B-operand TMA producer warp
// (non-halo kernels; the single producer warp needed ~620 clk of address arithmetic and issue per 2-k-block stage and
// was the critical path of the 64-wide low-resolution layers)
constexpr int kConvThreads = 224;
constexpr int kConvBWarp = 6;
constexpr int kXfWarps = 8;             // + 8 transform warps in the fused-GroupNorm variants (XF)
constexpr int kConvThreadsXf = kConvThreads + 32 * kXfWarps;
constexpr int kABytes = kConvBlockM * kConvBlockK * 2;  // 16 KB

// One persistent CTA per SM; STAGES x (A 16 KB + B) fills the ~190 KB of shared memory it can use, so
// enough TMA loads are in flight to cover the load round trip (small grids are latency-bound).
// PAIR: two CTAs of a cluster (an SM pair) run ONE tcgen05.mma.cta_group::2 of shape 256 x BN x 16: each CTA
// stages its own 128 output pixels of A and only HALF of the B tile, so a stage is 24 KB instead of 32 KB
// for the same tensor work - the main loop needs 25 % fewer bytes in flight / from L2 per FLOP.
// HALO (3x3, stride 1; always an SM pair): a CTA owns an (8*MT) x 16-pixel brick of one image (MT = 1 or 2 M tiles
// of 128 pixels).  ONE pipeline stage = one TMA load of the brick's (8*MT+2) x 16 halo for a given (horizontal tap,
// 64-channel chunk) + the three B tiles of its vertical taps; the vertical taps are 16-row (2 KB, swizzle-aligned)
// offsets into the same smem tile and the MT M tiles are 128-row offsets, so one mbarrier hand-shake feeds
// 3*MT*4 tcgen05.mma instead of 4.  Why: (1) the main loop of the plain kernel is bound by the ~45 B/clk/SM the
// L2 delivers (24 KB per 128x128x64 k-block = ~500 clk against 256 tensor clk); halo + pair needs 14.7 KB (MT=1) /
// 10 KB (MT=2, B shared by both M tiles); (2) clock64 traces show ~170 clk per mbarrier try_wait and ~30 clk per
// UTCHMMA issue in the single issuing warp - with one wait per k-block the issue loop itself costs ~400 clk.
constexpr int kHaloWt = 16, kHaloHt = 8;
// KPS (plain kernels): k-blocks per pipeline stage.  The single-warp producer / MMA loops cost ~450 clk per
// hand-shake (try_wait ~100-170, expect_tx + 2 TMA issues ~150, tcgen05.commit ~100); small grids are bound by
// exactly that (a 128x64x64 k-block is 128 tensor clk), so they put 2 k-blocks behind one barrier.
template <int BN, int STAGES, bool PAIR = false, bool HALO = false, int MT = 1, int KPS = 1>
struct ConvCfg {
  static_assert(!HALO || KPS == 1, "halo stages are already fused");
  static constexpr int kKps = KPS;
  static constexpr int kKbBytes = kABytes + ((PAIR ? BN / 2 : BN) * kConvBlockK * 2 + 1023) / 1024 * 1024;   // [A][B]
  static_assert(!HALO || (PAIR && (BN == 128 || BN == 16)), "halo kernels are SM-pair kernels with 128- or 16-wide N tiles");
  static constexpr int kMt = MT;
  static constexpr int kBRows = PAIR ? BN / 2 : BN;             // B rows staged by this CTA
  static constexpr int kBBytes = kBRows * kConvBlockK * 2;
  static constexpr int kBBytesPad = (kBBytes + 1023) / 1024 * 1024;
  static constexpr int kHaloABytes = (kHaloHt * MT + 2) * kHaloWt * 128;   // 20 KB (MT=1) / 36 KB (MT=2)
  // non-halo: [A 16 KB][B]; halo: [A halo][B kh=0][B kh=1][B kh=2]
  static constexpr int kStageBytes = HALO ? kHaloABytes + 3 * kBBytesPad : KPS * kKbBytes;
  static constexpr int kRingBytes = STAGES * kStageBytes;
  static constexpr int kStages = STAGES;
  static constexpr int kAccCols = BN * MT;                      // one accumulator buffer
  static constexpr int kTmemCols = 2 * kAccCols < 32 ? 32 : 2 * kAccCols;   // double-buffered accumulator
  static constexpr int kSlabs = BN / 64;                        // 64-channel output slabs (0: fp32 NCHW path)
  static constexpr int kStagingBytes = kSlabs * kConvBlockM * 128;
  static constexpr int kRedBytes = kSlabs > 0 ? 8192 : 0;       // GroupNorm-statistics scratch [row groups][BN][2]
  static constexpr int kSmemBytes = kRingBytes + kStagingBytes + kRedBytes + 1024 /*align*/ + 512 /*barriers*/;
  static_assert((3 * STAGES + 6) * 8 + 8 <= 512, "barrier block");
};

struct ConvKParams {
  int N, Ho, Wo, Cout;
  int Wt, Ht, Nt, w_blks, h_blks;
  int taps, c0_chunks, c1_chunks, r0_chunks, r1_chunks;
  int tap_dc[9], tap_dw[9], tap_da[9], tap_dh[9];
  int b_batch_rows;         // rows of B per image (attention GEMMs), 0 for shared weights
  int debug;                // B2E_DEBUG micro-benchmark knobs: 1 = no TMA loads (MMA on stale smem), 2 = no MMAs
  int splits;               // split-K factor (>1: partial accumulators meet in split_ws, last CTA finishes the tile)
  int split_cluster;        // 1: the splits of a tile form a thread-block cluster; partials meet in the leader's smem (DSMEM)
  // halo kernels: taps served per halo load (vertical) / loads per channel chunk (horizontal) and the offset of the
  // halo's first pixel from the brick's: 3, 3, (-1, -1) for a 3x3 convolution; 2, 2, (a - 1, b - 1) for sub-pixel phase (a, b)
  int halo_vt, halo_ht, halo_dh0, halo_dw0;
  float* split_ws;          // [num_tiles][splits][128][BN] fp32
  int* split_counters;      // [num_tiles], zero between launches
  int n_tiles, num_tiles;   // PAIR kernels: num_tiles counts tile PAIRS (two adjacent M tiles, same N tile)
  const float* bias;
  const float* bias2;
  const float* temb;
  int temb_stride;
  int out_f16;         // 1: stage + TMA-store the f16 NHWC tile through map_out
  float* out_f32_nchw;
  float* tile_stats;    // fused GroupNorm statistics or null
  int relu;             // 1: ReLU before the f16 store (classifier network)
  float acc_scale;      // accumulator * acc_scale before bias (weights packed with a power-of-two scale), 1: none
  // XF kernels: fused GroupNorm(+SiLU) of the A operand.  The TMA lands the RAW activation tile; the transform warps
  // rewrite it in shared memory as f16(silu(x * scale[n][c] + shift[n][c])) (zero where the convolution pads) before the
  // MMA warp sees it.  gn_coef = (scale, shift) per (image, K position of the concatenated sources), from gn_coeffs_kernel
  const float2* gn_coef; int coef_stride; int gn_silu; int Hin, Win;
  int split_pitch;      // > 0: split-f16 output (fp32-accurate mode): planes [hi | lo | hi] of split_pitch channels each
  long long* trace;     // B2E_TRACE: clock64 stamps of CTA 0's warp loops (halo kernels), else null
};
// trace regions (long long indices): MMA [0, 4*512) {iter start, A ready, B ready, issued}; producer A
// [2048, +3*256) {start, slot free, issued}; producer B [2816, +3*512); epilogue [4352, +4*64) {start, acc full, tmem released, done}
constexpr int kConvMaxSplits = 8;   // split-K factor bound (the finishing CTA keeps one load per split in flight)
// cluster split-K (64-wide N tiles): the leader's 192 KB ring holds the 6 other splits' 32 KB partial tiles
constexpr int kConvMaxClusterSplits = 7;
int conv_cluster_split_capacity(int splits);   // co-resident clusters of `splits` CTAs of the 64-wide kernel (0: cannot launch)
constexpr int kTrMma = 0, kTrPa = 2048, kTrPb = 2816, kTrEpi = 4352, kTrTotal = 4608;
// per-CTA wall clock (%globaltimer, ns): [kTrCta + 4 b + {0 entry, 1 after the prologue / grid dependency, 2 exit, 3 last split}]
constexpr int kTrCta = kTrTotal, kTrCtaMax = 160, kTrAll = kTrTotal + 8 * kTrCtaMax;
__device__ __forceinline__ long long global_ns() { long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }

// ------------------------------------------------------------------ the kernel
// Persistent: one CTA per SM walks tiles blockIdx.x, blockIdx.x + gridDim.x, ...  The accumulator is
// double-buffered in TMEM (2 x BN columns) so the epilogue of tile i overlaps the main loop of tile
// i+1, and the TMA producer runs ahead across tile boundaries (the smem ring never drains).
struct TileCoord { int n_tile, m_tile, w0, h0, n0; };

// pair kernels: `tile` indexes a pair of adjacent M tiles; this CTA takes M tile 2*(tile / n_tiles) + rank
__device__ __forceinline__ TileCoord tile_coord(const ConvKParams& p, int tile, int pair = 0, int rank = 0) {
  TileCoord t;
  t.n_tile = tile % p.n_tiles;
  int m = tile / p.n_tiles;
  if (pair) m = 2 * m + rank;
  t.m_tile = m;
  t.w0 = (m % p.w_blks) * p.Wt; m /= p.w_blks;
  t.h0 = (m % p.h_blks) * p.Ht;
  t.n0 = (m / p.h_blks) * p.Nt;
  return t;
}
// halo kernels: the work item of a CTA is a brick of MT vertically adjacent 8x16 tiles of one image;
// (w0, h0) = the brick's first pixel, m_tile = the statistics slot of its FIRST tile (tile mt: + mt * w_blks)
template <int MT>
__device__ __forceinline__ TileCoord halo_coord(const ConvKParams& p, int tile, int rank) {
  TileCoord t;
  t.n_tile = tile % p.n_tiles;
  int m = 2 * (tile / p.n_tiles) + rank;
  const int wb = m % p.w_blks; m /= p.w_blks;
  const int hbricks = p.h_blks / MT;
  const int hb = (m % hbricks) * MT;
  t.n0 = m / hbricks;
  t.w0 = wb * kHaloWt; t.h0 = hb * kHaloHt;
  t.m_tile = (t.n0 * p.h_blks + hb) * p.w_blks + wb;
  return t;
}

template <int BN, int STAGES, bool PAIR, bool HALO, int MT, int KPS, bool XF>
__global__ void __launch_bounds__(XF ? kConvThreadsXf : kConvThreads, 1)
conv_igemm_kernel(const __grid_constant__ CUtensorMap map_a0, const __grid_constant__ CUtensorMap map_a1,
                  const __grid_constant__ CUtensorMap map_r0, const __grid_constant__ CUtensorMap map_r1,
                  const __grid_constant__ CUtensorMap map_b, const __grid_constant__ CUtensorMap map_out,
                  const __grid_constant__ ConvKParams p) {
  using Cfg = ConvCfg<BN, STAGES, PAIR, HALO, MT, KPS>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* staging = smem + Cfg::kRingBytes;
  float* red = reinterpret_cast<float*>(staging + Cfg::kStagingBytes);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(staging + Cfg::kStagingBytes + Cfg::kRedBytes);
  uint64_t* empty_bar = full_bar + Cfg::kStages;
  uint64_t* tmem_full_bar = empty_bar + Cfg::kStages;   // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;         // [2]
  // XF: the A tile of a stage completes on THIS CTA's araw_bar (raw activations landed); the transform warps then
  // rewrite it and arrive on the (leader's) full_bar, which also collects the B tile's TMA bytes as before
  uint64_t* araw_bar = tmem_empty_bar + 2;              // [STAGES]
  // cluster split-K: part_bar (leader) collects the other splits' partial tiles, go_bar (others) = "the leader's ring is free"
  uint64_t* part_bar = araw_bar + Cfg::kStages;
  uint64_t* go_bar = part_bar + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(go_bar + 1);
  volatile uint32_t* split_flag = tmem_slot + 1;

  // warp index / cluster rank through shfl so that the compiler can prove them warp-uniform: the role branches
  // are then convergent and the producer / MMA loops keep coordinates, descriptors and barrier addresses in
  // uniform registers (otherwise every UTMALDG is preceded by ELECT + up to nine R2UR.BROADCAST, ~180 clk per TMA)
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  if (p.trace && blockIdx.x == 0 && threadIdx.x == 0) p.trace[kTrTotal - 1] = clock64();   // kernel entry
  if (p.trace && blockIdx.x < kTrCtaMax && threadIdx.x == 0) p.trace[kTrCta + 8 * blockIdx.x] = global_ns();
  const int rank = PAIR ? __shfl_sync(0xffffffffu, (int)cluster_ctarank(), 0) : 0;      // 0 = leader CTA of the SM pair
  const int tile_begin = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int tile_step = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int chunks = p.c0_chunks + p.c1_chunks;
  const int r_chunks = p.r0_chunks + p.r1_chunks;
  const int num_kb = p.taps * chunks + r_chunks;
  const int main_kb = p.taps * chunks;
  // work item = (tile, K split); consecutive CTAs take the splits of one tile
  const int splits = PAIR ? 1 : p.splits;
  const int num_work = p.num_tiles * splits;
  // cluster split-K (host: grid == num_work, cluster = the `splits` consecutive CTAs of one tile, split == cluster rank)
  const bool cl_split = !PAIR && !HALO && p.split_cluster != 0;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&map_a0);
    if (p.c1_chunks) prefetch_tmap(&map_a1);
    if (p.r0_chunks) prefetch_tmap(&map_r0);
    if (p.r1_chunks) prefetch_tmap(&map_r1);
    prefetch_tmap(&map_b);
    if (p.out_f16) prefetch_tmap(&map_out);
    for (int s = 0; s < Cfg::kStages; ++s) {
      // non-halo: one arrival per producer warp (A, B); XF: the A tile arrives through the transform warps instead
      mbar_init(full_bar + s, XF ? 1 + kXfWarps * (PAIR ? 2 : 1) : (HALO ? 1 : 2));
      mbar_init(empty_bar + s, 1);
      mbar_init(araw_bar + s, 1);
    }
    // pair: the leader's tmem_empty barrier collects the 4 epilogue warps of BOTH CTAs
    for (int s = 0; s < 2; ++s) { mbar_init(tmem_full_bar + s, 1); mbar_init(tmem_empty_bar + s, PAIR ? 8 : 4); }
    mbar_init(part_bar, 1);
    mbar_init(go_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    if (PAIR) tmem_alloc_2sm<Cfg::kTmemCols>(tmem_slot); else tmem_alloc<Cfg::kTmemCols>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR || cl_split) cluster_sync_all();   // peer barriers are initialised before any remote arrive / TMA completion
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // everything above touched only parameters and shared / tensor memory: from here on the previous kernel's
  // outputs are read (activations through TMA, time embedding in the epilogue)
  pdl_wait();
  pdl_trigger();
  if (p.trace && blockIdx.x < kTrCtaMax && threadIdx.x == 0) p.trace[kTrCta + 8 * blockIdx.x + 1] = global_ns();

  if (warp == 0) {
    // ===== TMA producer (whole warp walks the loop; one elected lane issues)
    int stage = 0; uint32_t phase = 0;
    if constexpr (HALO) {
      int tr_n = 0;
      const bool tr = p.trace && blockIdx.x == 0 && lane == 0;
      for (int tile = tile_begin; tile < p.num_tiles; tile += tile_step) {
        const TileCoord tc = halo_coord<MT>(p, tile, rank);
        const int brow0 = tc.n_tile * BN + rank * Cfg::kBRows;
        const int groups = p.halo_ht * chunks + r_chunks;
        const uint32_t a_bytes = (uint32_t)((kHaloHt * MT + p.halo_vt - 1) * kHaloWt * 128);   // the TMA box of the halo
        int kw = 0, ck = 0;
        for (int g = 0; g < groups; ++g) {
          const bool main = g < p.halo_ht * chunks;
          if (tr && tr_n < 512) p.trace[kTrPb + tr_n * 3] = clock64();
          mbar_wait(empty_bar + stage, phase ^ 1);
          if (tr && tr_n < 512) p.trace[kTrPb + tr_n * 3 + 1] = clock64();
          uint8_t* sa = smem + stage * Cfg::kStageBytes;
          if (elect_one()) {
            if (main) {
              // (8*MT+2) x 16 halo brick of horizontal tap kw + the B tiles of its three vertical taps
              const bool first = ck < p.c0_chunks;
              if constexpr (XF) {
                // raw activations: completion on this CTA's own barrier, the transform warps take it from there
                mbar_expect_tx(araw_bar + stage, a_bytes);
                tma_load_5d(sa, first ? &map_a0 : &map_a1, araw_bar + stage,
                            (first ? ck : ck - p.c0_chunks) * kConvBlockK, tc.w0 + kw + p.halo_dw0, 0, tc.h0 + p.halo_dh0, tc.n0);
                if (rank == 0) mbar_expect_tx(full_bar + stage, 2 * p.halo_vt * Cfg::kBBytes);
              } else {
              if (rank == 0) mbar_expect_tx(full_bar + stage, 2 * (a_bytes + p.halo_vt * Cfg::kBBytes));
              tma_load_5d_2sm(sa, first ? &map_a0 : &map_a1, full_bar + stage,
                              (first ? ck : ck - p.c0_chunks) * kConvBlockK, tc.w0 + kw + p.halo_dw0, 0, tc.h0 + p.halo_dh0, tc.n0);
              }
#pragma unroll
              for (int kh = 0; kh < 3; ++kh)
                if (kh < p.halo_vt)
                  tma_load_2d_2sm(sa + Cfg::kHaloABytes + kh * Cfg::kBBytesPad, &map_b, full_bar + stage,
                                  ((kh * p.halo_ht + kw) * chunks + ck) * kConvBlockK, brow0);
            } else {
              // residual segment: the brick itself (MT x 128 pixels) at the output position, one B tile
              const int rk = g - p.halo_ht * chunks;
              const bool first = rk < p.r0_chunks;
              if constexpr (XF) {
                mbar_expect_tx(araw_bar + stage, MT * kABytes);
                tma_load_5d(sa, first ? &map_r0 : &map_r1, araw_bar + stage,
                            (first ? rk : rk - p.r0_chunks) * kConvBlockK, tc.w0, 0, tc.h0, tc.n0);
                if (rank == 0) mbar_expect_tx(full_bar + stage, 2 * Cfg::kBBytes);
              } else {
              if (rank == 0) mbar_expect_tx(full_bar + stage, 2 * (MT * kABytes + Cfg::kBBytes));
              tma_load_5d_2sm(sa, first ? &map_r0 : &map_r1, full_bar + stage,
                              (first ? rk : rk - p.r0_chunks) * kConvBlockK, tc.w0, 0, tc.h0, tc.n0);
              }
              tma_load_2d_2sm(sa + Cfg::kHaloABytes, &map_b, full_bar + stage, (main_kb + rk) * kConvBlockK, brow0);
            }
          }
          __syncwarp();
          if (tr && tr_n < 512) { p.trace[kTrPb + tr_n * 3 + 2] = clock64(); ++tr_n; }
          if (++ck == chunks) { ck = 0; ++kw; }
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
        }
      }
    } else {
      // a stage = KPS k-blocks, each this CTA's A brick + its share of the B tile (pair: both CTAs complete on the
      // leader's barrier)
      int tr_n = 0;
      const bool tr = p.trace && blockIdx.x == 0 && lane == 0;
      for (int wi = tile_begin; wi < num_work; wi += tile_step) {
        const int tile = wi / splits, split = wi - tile * splits;
        const TileCoord tc = tile_coord(p, tile, PAIR, rank);
        const int kb0 = (int)((int64_t)split * num_kb / splits), kb1 = (int)((int64_t)(split + 1) * num_kb / splits);
        // walk (tap, chunk) incrementally: this warp sits on the critical path
        int tap = kb0 < main_kb ? kb0 / chunks : p.taps, ck = kb0 < main_kb ? kb0 - tap * chunks : kb0 - main_kb;
        int cw = 0, ch = 0, ca = 0, cc = 0;
        if (tap < p.taps) { cw = tc.w0 + p.tap_dw[tap]; ch = tc.h0 + p.tap_dh[tap]; ca = p.tap_da[tap]; cc = p.tap_dc[tap]; }
        for (int kb = kb0; kb < kb1; kb += KPS) {
          const int cnt = (kb1 - kb) < KPS ? (kb1 - kb) : KPS;   // k-blocks in this stage
          if (tr && tr_n < 512) p.trace[kTrPb + tr_n * 3] = clock64();
          mbar_wait(empty_bar + stage, phase ^ 1);
          if (tr && tr_n < 512) p.trace[kTrPb + tr_n * 3 + 1] = clock64();
          const bool leader = elect_one();
          if (leader) {
            if constexpr (XF) {
              mbar_expect_tx(araw_bar + stage, cnt * kABytes);
            } else {
            if (p.debug & 1) { if (rank == 0) mbar_arrive(full_bar + stage); }
            else if (!PAIR || rank == 0) mbar_expect_tx(full_bar + stage, (PAIR ? 2 : 1) * cnt * kABytes);
            }
          }
#pragma unroll
          for (int j = 0; j < KPS; ++j) {
            if (j < cnt) {
              const CUtensorMap* ma; int c0, c1, c2, c3;
              if (tap < p.taps) {
                const bool first = ck < p.c0_chunks;
                ma = first ? &map_a0 : &map_a1;
                c0 = cc + (first ? ck : ck - p.c0_chunks) * kConvBlockK; c1 = cw; c2 = ca; c3 = ch;
              } else {   // residual segment: 1x1 at the output pixel
                const bool first = ck < p.r0_chunks;
                ma = first ? &map_r0 : &map_r1;
                c0 = (first ? ck : ck - p.r0_chunks) * kConvBlockK; c1 = tc.w0; c2 = 0; c3 = tc.h0;
              }
              if (leader && !(p.debug & 1)) {
                uint8_t* sa = smem + stage * Cfg::kStageBytes + j * Cfg::kKbBytes;
                if (PAIR) {
                  if constexpr (XF) tma_load_5d(sa, ma, araw_bar + stage, c0, c1, c2, c3, tc.n0);
                  else tma_load_5d_2sm(sa, ma, full_bar + stage, c0, c1, c2, c3, tc.n0);
                } else {
                  tma_load_5d(sa, ma, (XF ? araw_bar : full_bar) + stage, c0, c1, c2, c3, tc.n0);
                }
              }
              ++ck;
              if (tap < p.taps && ck == chunks) {
                ck = 0;
                if (++tap < p.taps) { cw = tc.w0 + p.tap_dw[tap]; ch = tc.h0 + p.tap_dh[tap]; ca = p.tap_da[tap]; cc = p.tap_dc[tap]; }
              }
            }
          }
          __syncwarp();
          if (tr && tr_n < 512) { p.trace[kTrPb + tr_n * 3 + 2] = clock64(); ++tr_n; }
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (whole warp walks the loop; one elected lane issues)
    if (rank == 0) {   // pair: only the leader CTA issues (for both SMs)
      constexpr uint32_t idesc = make_idesc(PAIR ? 2 * kConvBlockM : kConvBlockM, BN);
      int stage = 0; uint32_t phase = 0;
      int it = 0;
      if constexpr (HALO) {
        int tr_n = 0;
        const bool tr = p.trace && blockIdx.x == 0 && lane == 0;
        const int groups = p.halo_ht * chunks + r_chunks;   // pipeline stages per work item
        for (int tile = tile_begin; tile < p.num_tiles; tile += tile_step, ++it) {
          const int acc = it & 1;
          if (tr && tr_n < 512) p.trace[kTrMma + tr_n * 4] = clock64();
          mbar_wait(tmem_empty_bar + acc, ((it >> 1) & 1) ^ 1);
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + (uint32_t)(acc * Cfg::kAccCols);
          for (int g = 0; g < groups; ++g) {
            const int nsub = g < p.halo_ht * chunks ? p.halo_vt : 1;   // vertical taps served by this stage
            if (tr && tr_n < 512) p.trace[kTrMma + tr_n * 4 + 1] = clock64();
            if constexpr (XF) mbar_wait_cluster(full_bar + stage, phase); else mbar_wait(full_bar + stage, phase);
            tc_fence_after();
            if (tr && tr_n < 512) p.trace[kTrMma + tr_n * 4 + 2] = clock64();
            const uint32_t a_addr = smem_u32(smem + stage * Cfg::kStageBytes);
            const uint32_t b_addr = a_addr + Cfg::kHaloABytes;
            if (elect_one()) {
#pragma unroll
              for (int mt = 0; mt < MT; ++mt) {
                for (int kh = 0; kh < nsub; ++kh) {
                  // M tile mt / vertical tap kh = rows [(8*mt + kh) * 16, + 128) of the halo tile (2 KB-aligned)
                  const uint64_t adesc = make_smem_desc(a_addr + (uint32_t)((mt * kHaloHt + kh) * kHaloWt * 128));
                  const uint64_t bdesc = make_smem_desc(b_addr + (uint32_t)(kh * Cfg::kBBytesPad));
#pragma unroll
                  for (int k = 0; k < kConvBlockK / 16; ++k)
                    umma_f16_2sm(tmem_d + (uint32_t)(mt * BN), adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc,
                                  (g == 0 && kh == 0 && k == 0) ? 0u : 1u);
                }
              }
              // frees this stage in both CTAs once the MMAs above retire
              umma_commit_2sm(empty_bar + stage);
              if (g == groups - 1) umma_commit_2sm(tmem_full_bar + acc);
            }
            __syncwarp();
            if (tr && tr_n < 512) { p.trace[kTrMma + tr_n * 4 + 3] = clock64(); ++tr_n; if (tr_n < 512) p.trace[kTrMma + tr_n * 4] = 0; }
            if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
          }
        }
      } else {
        int tr_n = 0;
        const bool tr = p.trace && blockIdx.x == 0 && lane == 0;
        for (int wi = tile_begin; wi < num_work; wi += tile_step, ++it) {
          const int split = wi % splits;
          const int kb0 = (int)((int64_t)split * num_kb / splits), kb1 = (int)((int64_t)(split + 1) * num_kb / splits);
          const int acc = it & 1;
          mbar_wait(tmem_empty_bar + acc, ((it >> 1) & 1) ^ 1);  // epilogue has drained this accumulator
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BN);
          for (int kb = kb0; kb < kb1; kb += KPS) {
            const int cnt = (kb1 - kb) < KPS ? (kb1 - kb) : KPS;
            if (tr && tr_n < 512) { p.trace[kTrMma + tr_n * 4] = p.trace[kTrMma + tr_n * 4 + 1] = clock64(); }
            if constexpr (XF) mbar_wait_cluster(full_bar + stage, phase); else mbar_wait(full_bar + stage, phase);
            tc_fence_after();
            if (tr && tr_n < 512) p.trace[kTrMma + tr_n * 4 + 2] = clock64();
            const uint32_t sbase = smem_u32(smem + stage * Cfg::kStageBytes);
            if (elect_one()) {
#pragma unroll
              for (int j = 0; j < KPS; ++j) {
                if (j < cnt && !(p.debug & 2)) {
                  const uint64_t adesc = make_smem_desc(sbase + j * Cfg::kKbBytes);
                  const uint64_t bdesc = make_smem_desc(sbase + j * Cfg::kKbBytes + kABytes);
#pragma unroll
                  for (int k = 0; k < kConvBlockK / 16; ++k) {
                    // advance 16 f16 = 32 B along K inside the swizzle row: +2 in the (addr >> 4) field
                    const uint32_t accum = (kb > kb0 || j > 0 || k > 0) ? 1u : 0u;
                    if (PAIR) umma_f16_2sm(tmem_d, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, accum);
                    else umma_f16(tmem_d, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, accum);
                  }
                }
              }
              // frees this smem stage (in both CTAs of a pair) once the MMAs above retire
              if (PAIR) umma_commit_2sm(empty_bar + stage); else umma_commit(empty_bar + stage);
              // accumulator complete (pair: rows 0-127 in the leader's TMEM, 128-255 in the peer's)
              if (kb + KPS >= kb1) { if (PAIR) umma_commit_2sm(tmem_full_bar + acc); else umma_commit(tmem_full_bar + acc); }
            }
            __syncwarp();
            if (tr && tr_n < 512) { p.trace[kTrMma + tr_n * 4 + 3] = clock64(); ++tr_n; }
            if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == kConvBWarp) {
    // ===== B-operand TMA producer (non-halo kernels): same stage walk as warp 0, one 2D load of the weight tile per k-block
    if constexpr (!HALO) {
      int stage = 0; uint32_t phase = 0;
      for (int wi = tile_begin; wi < num_work; wi += tile_step) {
        const int tile = wi / splits, split = wi - tile * splits;
        const TileCoord tc = tile_coord(p, tile, PAIR, rank);
        // per-image B rows for batched GEMMs (Nt == 1); pair: this CTA's half of the N tile
        const int brow0 = tc.n_tile * BN + tc.n0 * p.b_batch_rows + (PAIR ? rank * Cfg::kBRows : 0);
        const int kb0 = (int)((int64_t)split * num_kb / splits), kb1 = (int)((int64_t)(split + 1) * num_kb / splits);
        for (int kb = kb0; kb < kb1; kb += KPS) {
          const int cnt = (kb1 - kb) < KPS ? (kb1 - kb) : KPS;
          mbar_wait(empty_bar + stage, phase ^ 1);
          if (elect_one()) {
            if (p.debug & 1) { if (!XF && rank == 0) mbar_arrive(full_bar + stage); }
            else {
              if (!PAIR || rank == 0) mbar_expect_tx(full_bar + stage, (PAIR ? 2 : 1) * cnt * Cfg::kBBytes);
#pragma unroll
              for (int j = 0; j < KPS; ++j) {
                if (j < cnt) {
                  uint8_t* sb = smem + stage * Cfg::kStageBytes + j * Cfg::kKbBytes + kABytes;
                  if (PAIR) tma_load_2d_2sm(sb, &map_b, full_bar + stage, (kb + j) * kConvBlockK, brow0);
                  else tma_load_2d(sb, &map_b, full_bar + stage, (kb + j) * kConvBlockK, brow0);
                }
              }
            }
          }
          __syncwarp();
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp < kConvBWarp) {
    // ===== epilogue: 4 warps, warp w owns TMEM lanes 32*(w%4) .. +31
    const int q = warp & 3;
    const int r = q * 32 + lane;  // row of the tile = output pixel
    const int w_l = r % p.Wt, h_l = (r / p.Wt) % p.Ht, n_l = r / (p.Wt * p.Ht);
    const bool store_leader = (warp == 2 && lane == 0);
    int it = 0;
    for (int wi = tile_begin; wi < num_work; wi += tile_step, ++it) {
      const int tile = wi / splits, split = wi - tile * splits;
      const TileCoord tc0 = HALO ? halo_coord<MT>(p, tile, rank) : tile_coord(p, tile, PAIR, rank);
      const int acc = it & 1;
      const bool tr = p.trace && blockIdx.x == 0 && threadIdx.x == 64 && it < 64;
      if (tr) p.trace[kTrEpi + it * 4] = clock64();
      mbar_wait(tmem_full_bar + acc, (it >> 1) & 1);
      tc_fence_after();
      if (tr) p.trace[kTrEpi + it * 4 + 1] = clock64();
#pragma unroll 1
      for (int mt = 0; mt < MT; ++mt) {   // halo kernels: the MT M tiles of the brick, one after the other
      TileCoord tc = tc0;
      tc.h0 += mt * kHaloHt; tc.m_tile += mt * p.w_blks;
      const int n = tc.n0 + n_l, h = tc.h0 + h_l, w = tc.w0 + w_l;
      const bool valid = n < p.N;
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * Cfg::kAccCols + mt * BN);
      auto release_tmem = [&]() {
        if (mt != MT - 1) return;
        // all of this warp's accumulator columns are in registers: hand the buffer back
        tc_fence_before();
        __syncwarp();
        if (lane == 0) { if (PAIR) mbar_arrive_leader(tmem_empty_bar + acc); else mbar_arrive(tmem_empty_bar + acc); }
        if (tr) p.trace[kTrEpi + it * 4 + 2] = clock64();
      };
      const float* part_row = nullptr;
      const float* part_smem = nullptr;
      if (splits > 1 && cl_split) {
        // cluster split-K: the splits of this tile are the CTAs of one cluster.  Every other split parks its raw fp32
        // accumulator in its OWN (drained) smem ring as [16-col chunk][float4 j][row][4] and, once the leader's ring is
        // free too, bulk-copies it into the leader's ring (DSMEM, completes on the leader's part_bar); the leader sums
        // own accumulator + partials in split order and runs the normal epilogue.  No global workspace, fence or atomics.
        constexpr uint32_t kPartBytes = kConvBlockM * BN * sizeof(float);
        if (split != 0) {
          float* mine = reinterpret_cast<float*>(smem);
#pragma unroll 1
          for (int c = 0; c < BN / 16; ++c) {
            float v[16];
            tmem_ld16(taddr + c * 16, v);
            if (c == BN / 16 - 1) release_tmem();
#pragma unroll
            for (int j = 0; j < 4; ++j)
              *reinterpret_cast<float4*>(mine + ((c * 4 + j) * kConvBlockM + r) * 4) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          }
          fence_async_smem();
          epi_bar_sync();
          if (store_leader) {
            mbar_wait_cluster(go_bar, 0);
            bulk_copy_to_cluster(mapa_shared(smem_u32(smem) + (uint32_t)(split - 1) * kPartBytes, 0), smem_u32(smem), kPartBytes,
                                 mapa_shared(smem_u32(part_bar), 0));
          }
          continue;
        }
        if (warp == 2) {
          // this CTA's MMAs have retired (tmem_full): its ring is free.  One lane per other split signals it (in parallel:
          // a serial loop of release-arrives costs ~0.17 us per split)
          if (lane == 0) mbar_expect_tx(part_bar, (uint32_t)(splits - 1) * kPartBytes);
          __syncwarp();
          if (lane >= 1 && lane < splits) mbar_arrive_remote_release(mapa_shared(smem_u32(go_bar), (uint32_t)lane));
        }
        mbar_wait_cluster(part_bar, 0);
        part_smem = reinterpret_cast<const float*>(smem);
        if (p.trace && blockIdx.x < kTrCtaMax && store_leader) p.trace[kTrCta + 8 * blockIdx.x + 3] = global_ns();
      } else if (splits > 1) {
        // split-K: park the raw fp32 partial tile; the CTA that arrives last sums all partials (fixed order) and
        // runs the normal epilogue - no extra kernel, deterministic result
        // layout [tile][split][16-col chunk][row][16]: a warp's 32 rows write / read 2 KB contiguous
        float* mine = p.split_ws + ((int64_t)tile * splits + split) * (kConvBlockM * BN) + r * 16;
#pragma unroll 1
        for (int c = 0; c < BN / 16; ++c) {
          float v[16];
          tmem_ld16(taddr + c * 16, v);
          if (c == BN / 16 - 1) release_tmem();
#pragma unroll
          for (int j = 0; j < 4; ++j)
            __stcg(reinterpret_cast<float4*>(mine + c * (kConvBlockM * 16)) + j,
                   make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
        }
        __threadfence();
        epi_bar_sync();
        if (store_leader) {
          const int old = atomicAdd(p.split_counters + tile, 1);
          const bool last = old == splits - 1;
          if (last) p.split_counters[tile] = 0;   // every split has arrived: re-arm for the next launch
          *split_flag = last ? 1u : 0u;
        }
        epi_bar_sync();
        if (!*split_flag) continue;
        __threadfence();
        if (p.trace && blockIdx.x < kTrCtaMax && store_leader) p.trace[kTrCta + 8 * blockIdx.x + 3] = global_ns();
        part_row = p.split_ws + (int64_t)tile * splits * (kConvBlockM * BN) + r * 16;
      }
      // split-f16 output (fp32-accurate mode): the accumulator is walked twice - pass 0 stages f16(v) (planes 0 and
      // 2 of the output), pass 1 the remainder f16(v - f16(v)) (plane 1); TMEM is released after the last pass
      const int npass = (Cfg::kSlabs > 0 && p.out_f16 && p.split_pitch) ? 2 : 1;
#pragma unroll 1
      for (int pass = 0; pass < npass; ++pass) {
      if (Cfg::kSlabs > 0 && p.out_f16) {
        // the previous tile's TMA store must have finished reading the staging buffer
        if (store_leader) tma_store_wait_read();
        epi_bar_sync();
      }
      // Fast path (f16 NHWC output straight from TMEM, BN >= 32): 32 accumulator columns per iteration - both tcgen05.ld
      // and every bias / shortcut-bias / time-embedding load of the iteration are issued BEFORE the single wait, so their
      // latencies overlap (the 16-column loop below paid a TMEM round trip plus an L1 round trip eight times per tile:
      // ~4 500 clk per 128 x 128 tile, which made the K-short layers epilogue-bound - ncu tensor pipe 74 % at Cin 128).
      // Same arithmetic, same order of the adds.
      bool fast_done = false;
      if constexpr (Cfg::kSlabs > 0) {
        if (p.out_f16 && !part_row) {
          fast_done = true;
#pragma unroll 1
          for (int c2 = 0; c2 < BN / 32; ++c2) {
            uint32_t raw[32];
            tmem_ld16_issue(taddr + c2 * 32, raw);
            tmem_ld16_issue(taddr + c2 * 32 + 16, raw + 16);
            const int col0 = tc.n_tile * BN + c2 * 32;
            float4 b1[8], b2[8], tb[8];
            const bool hb1 = p.bias != nullptr, hb2 = p.bias2 != nullptr, htb = p.temb != nullptr && valid;
            if (hb1) {
              const float4* bp = reinterpret_cast<const float4*>(p.bias + col0);
#pragma unroll
              for (int j = 0; j < 8; ++j) b1[j] = __ldg(bp + j);
            }
            if (hb2) {
              const float4* bp = reinterpret_cast<const float4*>(p.bias2 + col0);
#pragma unroll
              for (int j = 0; j < 8; ++j) b2[j] = __ldg(bp + j);
            }
            if (htb) {
              const float4* tp = reinterpret_cast<const float4*>(p.temb + (int64_t)n * p.temb_stride + col0);
#pragma unroll
              for (int j = 0; j < 8; ++j) tb[j] = __ldg(tp + j);
            }
            tmem_ld_wait();
            if (c2 == BN / 32 - 1 && pass == npass - 1) release_tmem();
            float v[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(raw[j]);
            if (part_smem) {
              // cluster split-K leader: own accumulator (split 0) + the other splits' partial tiles, in split order
              for (int sp = 1; sp < splits; ++sp) {
                const float* pp = part_smem + (int64_t)(sp - 1) * (kConvBlockM * BN) + (c2 * 8 * kConvBlockM + r) * 4;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  const float4 b = *reinterpret_cast<const float4*>(pp + j * kConvBlockM * 4);
                  v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
                }
              }
            }
            if (p.acc_scale != 1.f) {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] *= p.acc_scale;
            }
            if (hb1) {
#pragma unroll
              for (int j = 0; j < 8; ++j) { v[4 * j] += b1[j].x; v[4 * j + 1] += b1[j].y; v[4 * j + 2] += b1[j].z; v[4 * j + 3] += b1[j].w; }
            }
            if (hb2) {
#pragma unroll
              for (int j = 0; j < 8; ++j) { v[4 * j] += b2[j].x; v[4 * j + 1] += b2[j].y; v[4 * j + 2] += b2[j].z; v[4 * j + 3] += b2[j].w; }
            }
            if (htb) {
#pragma unroll
              for (int j = 0; j < 8; ++j) { v[4 * j] += tb[j].x; v[4 * j + 1] += tb[j].y; v[4 * j + 2] += tb[j].z; v[4 * j + 3] += tb[j].w; }
            }
            if (p.relu) {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
            }
            if (pass) {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = __fsub_rn(v[j], f16_to_float(float_to_f16(v[j])));
            }
            // 128B-swizzled staging tile: row r, 16-byte chunk j stored at chunk (j ^ (r & 7)); 32 columns = 4 chunks
            uint8_t* row = staging + (c2 >> 1) * (kConvBlockM * 128) + r * 128;
            const int j0 = (c2 & 1) * 4;
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4) {
              uint4 o;
              f16x2* ob = reinterpret_cast<f16x2*>(&o);
#pragma unroll
              for (int j = 0; j < 4; ++j) ob[j] = floats_to_f16x2(v[8 * k4 + 2 * j], v[8 * k4 + 2 * j + 1]);
              *reinterpret_cast<uint4*>(row + (((j0 + k4) ^ (r & 7)) << 4)) = o;
            }
          }
        }
      }
#pragma unroll 1
      for (int c = 0; c < (fast_done ? 0 : BN / 16); ++c) {
        float v[16];
        if (part_row) {
          // sum of the partial tiles in split order (deterministic).  The loads of ALL splits of an 8-column half are
          // issued before the first add - unconditionally, from a clamped split index, so that no branch keeps the
          // compiler from hoisting them: one L2 round trip per half.  (A per-split loop, and also predicated loads,
          // compile to one dependent round trip per split: 64 per tile, 12 of the 18 us of a low-resolution launch.)
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = 0.f;
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            float4 b[kConvMaxSplits][2];
#pragma unroll
            for (int sp = 0; sp < kConvMaxSplits; ++sp) {
              const int spc = sp < splits ? sp : 0;
              const float4* pp = reinterpret_cast<const float4*>(part_row + (int64_t)spc * (kConvBlockM * BN) + c * (kConvBlockM * 16)) + 2 * hh;
              if (p.debug & 16) { b[sp][0] = b[sp][1] = make_float4(0.f, 0.f, 0.f, 0.f); }
              else if (p.debug & 32) { b[sp][0] = *pp; b[sp][1] = *(pp + 1); }
              else { b[sp][0] = __ldcg(pp); b[sp][1] = __ldcg(pp + 1); }
            }
#pragma unroll
            for (int sp = 0; sp < kConvMaxSplits; ++sp) {
              const bool on = sp < splits;
              v[8 * hh] = on ? v[8 * hh] + b[sp][0].x : v[8 * hh];
              v[8 * hh + 1] = on ? v[8 * hh + 1] + b[sp][0].y : v[8 * hh + 1];
              v[8 * hh + 2] = on ? v[8 * hh + 2] + b[sp][0].z : v[8 * hh + 2];
              v[8 * hh + 3] = on ? v[8 * hh + 3] + b[sp][0].w : v[8 * hh + 3];
              v[8 * hh + 4] = on ? v[8 * hh + 4] + b[sp][1].x : v[8 * hh + 4];
              v[8 * hh + 5] = on ? v[8 * hh + 5] + b[sp][1].y : v[8 * hh + 5];
              v[8 * hh + 6] = on ? v[8 * hh + 6] + b[sp][1].z : v[8 * hh + 6];
              v[8 * hh + 7] = on ? v[8 * hh + 7] + b[sp][1].w : v[8 * hh + 7];
            }
          }
        } else {
          tmem_ld16(taddr + c * 16, v);
          if (c == BN / 16 - 1 && pass == npass - 1) release_tmem();
        }
        const int col0 = tc.n_tile * BN + c * 16;
        if (p.acc_scale != 1.f) {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] *= p.acc_scale;
        }
        if (Cfg::kSlabs > 0 && p.out_f16) {
          // Cout % 64 == 0 on this path (host-checked): whole chunks are in range
          if (p.bias) {
            const float4* bp = reinterpret_cast<const float4*>(p.bias + col0);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float4 b = __ldg(bp + j);
              v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
            }
          }
          if (p.bias2) {
            const float4* bp = reinterpret_cast<const float4*>(p.bias2 + col0);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float4 b = __ldg(bp + j);
              v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
            }
          }
          if (p.temb && valid) {
            const float4* tp = reinterpret_cast<const float4*>(p.temb + (int64_t)n * p.temb_stride + col0);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float4 b = __ldg(tp + j);
              v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
            }
          }
          if (p.relu) {
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
          }
          if (pass) {
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = __fsub_rn(v[j], f16_to_float(float_to_f16(v[j])));
          }
          uint4 o0, o1;
          f16x2* ob0 = reinterpret_cast<f16x2*>(&o0);
          f16x2* ob1 = reinterpret_cast<f16x2*>(&o1);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            ob0[j] = floats_to_f16x2(v[2 * j], v[2 * j + 1]);
            ob1[j] = floats_to_f16x2(v[8 + 2 * j], v[8 + 2 * j + 1]);
          }
          // 128B-swizzled staging tile: row r, 16-byte chunk j stored at chunk (j ^ (r & 7))
          uint8_t* row = staging + (c >> 2) * (kConvBlockM * 128) + r * 128;
          const int j0 = (c & 3) * 2;
          *reinterpret_cast<uint4*>(row + (((j0) ^ (r & 7)) << 4)) = o0;
          *reinterpret_cast<uint4*>(row + (((j0 + 1) ^ (r & 7)) << 4)) = o1;
        } else if (p.out_f32_nchw && valid) {
          const int64_t hw = (int64_t)p.Ho * p.Wo;
#pragma unroll
          for (int j = 0; j < 16; ++j)
            if (col0 + j < p.Cout) {
              float o = v[j];
              if (p.bias) o += __ldg(p.bias + col0 + j);
              if (p.bias2) o += __ldg(p.bias2 + col0 + j);
              if (p.temb) o += __ldg(p.temb + (int64_t)n * p.temb_stride + col0 + j);
              p.out_f32_nchw[((int64_t)n * p.Cout + col0 + j) * hw + (int64_t)h * p.Wo + w] = o;
            }
        }
      }
      if (p.trace && blockIdx.x < kTrCtaMax && store_leader && (part_row || part_smem)) p.trace[kTrCta + 8 * blockIdx.x + 4] = global_ns();
      if (Cfg::kSlabs > 0 && p.out_f16) {
        fence_async_smem();   // generic-proxy smem writes -> visible to the TMA (async proxy)
        epi_bar_sync();
        if (store_leader) {
#pragma unroll
          for (int sl = 0; sl < Cfg::kSlabs; ++sl) {
            const int ch = tc.n_tile * BN + sl * 64;
            tma_store_5d(&map_out, staging + sl * (kConvBlockM * 128), ch + pass * p.split_pitch, tc.w0, 0, tc.h0, tc.n0);
            if (p.split_pitch && pass == 0)
              tma_store_5d(&map_out, staging + sl * (kConvBlockM * 128), ch + 2 * p.split_pitch, tc.w0, 0, tc.h0, tc.n0);
          }
          tma_store_commit();
          if (p.trace && blockIdx.x < kTrCtaMax && (part_row || part_smem)) p.trace[kTrCta + 8 * blockIdx.x + 5] = global_ns();
        }
        if (p.tile_stats) {
          // GroupNorm statistics of the f16 tile just staged: per-channel sum / sum of squares over the
          // rows of each image in the tile (thread = 8 channels x a group of rows; deterministic order)
          constexpr int NC = BN / 8, NG = kConvBlockM / NC, RP = kConvBlockM / NG;
          const int t = threadIdx.x - 64;
          const int j = t % NC, g = t / NC;
          float sum[8], sq[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) sum[e] = sq[e] = 0.f;
#pragma unroll 4
          for (int rr = 0; rr < RP; ++rr) {
            const int row = g * RP + rr;
            const uint4 v = *reinterpret_cast<const uint4*>(staging + (j >> 3) * (kConvBlockM * 128) + row * 128 +
                                                            (((j & 7) ^ (row & 7)) << 4));
            const f16x2* b2 = reinterpret_cast<const f16x2*>(&v);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 f = f16x2_to_float2(b2[e]);
              sum[2 * e] += f.x; sq[2 * e] += f.x * f.x;
              sum[2 * e + 1] += f.y; sq[2 * e + 1] += f.y * f.y;
            }
          }
#pragma unroll
          for (int e = 0; e < 8; ++e)
            *reinterpret_cast<float2*>(red + ((g * BN) + j * 8 + e) * 2) = make_float2(sum[e], sq[e]);
          epi_bar_sync();
          if (t < BN) {
            const int groups_per_img = (p.Wt * p.Ht) / RP;
            for (int nl = 0; nl < p.Nt; ++nl) {
              float s1 = 0.f, s2 = 0.f;
              for (int gg = nl * groups_per_img; gg < (nl + 1) * groups_per_img; ++gg) {
                const float2 f = *reinterpret_cast<const float2*>(red + (gg * BN + t) * 2);
                s1 += f.x; s2 += f.y;
              }
              const int64_t slot = (int64_t)tc.m_tile * p.Nt + nl;
              *reinterpret_cast<float2*>(p.tile_stats + (slot * p.Cout + tc.n_tile * BN + t) * 2) = make_float2(s1, s2);
            }
          }
        }
      }
      }   // pass
      }   // mt
      if (tr) p.trace[kTrEpi + it * 4 + 3] = clock64();
    }
    if (store_leader) tma_store_wait_all();
    if (p.trace && blockIdx.x < kTrCtaMax && store_leader) p.trace[kTrCta + 8 * blockIdx.x + 6] = global_ns();
    tc_fence_before();
  } else {
    // ===== transform warps (XF): fused GroupNorm(+SiLU) of the A operand.  Per stage: wait for this CTA's raw tile
    // (araw_bar), rewrite it in place - thread = one 16-byte chunk column (8 channels) x every 32nd row, so its swizzled
    // chunk position and its 8 (scale, shift) pairs are fixed per k-block - zero the positions the convolution pads
    // (TMA filled them with raw zeros, which GroupNorm would turn into silu(shift)), make the writes visible to the
    // async proxy and arrive on the (leader's) full_bar.  Residual-segment stages pass through untouched.
    const int lt = (int)threadIdx.x - kConvThreads;
    const int cj = lt & 7, rr = lt >> 3;                     // chunk column, first row (rows rr + 32 i)
    const uint32_t swz = (uint32_t)((cj ^ (rr & 7)) << 4);   // (rr + 32 i) & 7 == rr & 7
    const bool silu = p.gn_silu != 0 && !(p.debug & 4);   // B2E_DEBUG micro-benchmark knobs: 4 = no SiLU, 8 = no rewrite at all
    const bool xf_skip = (p.debug & 8) != 0;
    int stage = 0; uint32_t phase = 0;
    auto xf_arrive = [&]() {
      fence_async_smem();
      __syncwarp();
      if (lane == 0) { if (PAIR) mbar_arrive_leader_release(full_bar + stage); else mbar_arrive(full_bar + stage); }
      if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
    };
    auto load_coef = [&](int n, int kpos, float* sc, float* sh) {
      const float4* cp = reinterpret_cast<const float4*>(p.gn_coef + (int64_t)n * p.coef_stride + kpos + cj * 8);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float4 v = __ldg(cp + e);
        sc[2 * e] = v.x; sh[2 * e] = v.y; sc[2 * e + 1] = v.z; sh[2 * e + 1] = v.w;
      }
    };
    if constexpr (HALO) {
      constexpr int kRows = (kHaloHt * MT + 2) * kHaloWt, kNI = kRows / 32;
      static_assert(kRows % 32 == 0, "halo rows");
      const int groups = p.halo_ht * chunks + r_chunks;
      for (int tile = tile_begin; tile < p.num_tiles; tile += tile_step) {
        const TileCoord tc = halo_coord<MT>(p, tile, rank);
        int kw = 0, ck = 0;
        for (int g = 0; g < groups; ++g) {
          const bool main = g < p.halo_ht * chunks;
          float sc[8], sh[8];
          if (main) load_coef(tc.n0, ck * kConvBlockK, sc, sh);     // before the wait: overlaps the TMA flight
          mbar_wait(araw_bar + stage, phase);
          if (main) {
            uint8_t* sa = smem + stage * Cfg::kStageBytes;
            const int wbase = tc.w0 + kw + p.halo_dw0, hbase = tc.h0 + p.halo_dh0;
            if (!xf_skip) {
#pragma unroll
              for (int i = 0; i < kNI; ++i) {
                const int r = rr + 32 * i;
                const int h = hbase + (r >> 4), w = wbase + (r & 15);
                uint4* ptr = reinterpret_cast<uint4*>(sa + r * 128 + swz);
                const bool in = (unsigned)h < (unsigned)p.Hin && (unsigned)w < (unsigned)p.Win;
                *ptr = in ? gn_apply8(*ptr, sc, sh, silu) : make_uint4(0, 0, 0, 0);
              }
            }
            if (++ck == chunks) { ck = 0; ++kw; }
          }
          xf_arrive();
        }
      }
    } else {
      // rows of the 128-pixel tile: r -> (image, row, column) within the Nt x Ht x Wt brick, fixed per thread
      int wl[4], hl[4], nl[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = rr + 32 * i;
        wl[i] = r % p.Wt; hl[i] = (r / p.Wt) % p.Ht; nl[i] = r / (p.Wt * p.Ht);
      }
      for (int wi = tile_begin; wi < num_work; wi += tile_step) {
        const int tile = wi / splits, split = wi - tile * splits;
        const TileCoord tc = tile_coord(p, tile, PAIR, rank);
        const int kb0 = (int)((int64_t)split * num_kb / splits), kb1 = (int)((int64_t)(split + 1) * num_kb / splits);
        for (int kb = kb0; kb < kb1; kb += KPS) {
          const int cnt = (kb1 - kb) < KPS ? (kb1 - kb) : KPS;
          mbar_wait(araw_bar + stage, phase);
#pragma unroll
          for (int j = 0; j < KPS; ++j) {
            const int k = kb + j;
            if (j < cnt && k < main_kb) {
              const int tap = k / chunks, ck = k - tap * chunks;
              const int dh = p.tap_dh[tap], dw = p.tap_dw[tap];
              uint8_t* sa = smem + stage * Cfg::kStageBytes + j * Cfg::kKbBytes;
              float sc[8], sh[8];
              int n_have = -1;
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const int r = rr + 32 * i;
                const int n = tc.n0 + nl[i], h = tc.h0 + hl[i] + dh, w = tc.w0 + wl[i] + dw;
                uint4* ptr = reinterpret_cast<uint4*>(sa + r * 128 + swz);
                const bool in = n < p.N && (unsigned)h < (unsigned)p.Hin && (unsigned)w < (unsigned)p.Win;
                if (in) {
                  if (n != n_have) { load_coef(n, ck * kConvBlockK, sc, sh); n_have = n; }
                  *ptr = gn_apply8(*ptr, sc, sh, silu);
                } else {
                  *ptr = make_uint4(0, 0, 0, 0);
                }
              }
            }
          }
          xf_arrive();
        }
      }
    }
  }
  __syncthreads();
  if (p.trace && blockIdx.x == 0 && threadIdx.x == 0) p.trace[kTrTotal - 2] = clock64();   // all roles done
  if (PAIR || cl_split) cluster_sync_all();   // no CTA leaves while its peer may still signal its barriers / read its smem
  if (warp == 1) {
    tc_fence_after();
    if (PAIR) tmem_dealloc_2sm<Cfg::kTmemCols>(tmem_base); else tmem_dealloc<Cfg::kTmemCols>(tmem_base);
  }
  if (p.trace && blockIdx.x < kTrCtaMax && threadIdx.x == 0) p.trace[kTrCta + 8 * blockIdx.x + 2] = global_ns();
}

// ------------------------------------------------------------------ weight packing
__global__ void pack_weight_kernel(const float* __restrict__ w, f16* __restrict__ out, int Cout, int Cin,
                                   int kk, int tap_width, int row_len, int col_off, int ci0, int cin_total, int lo,
                                   float wscale) {
  // out[co*row_len + col_off + t*tap_width + ci] = w[(co*cin_total + ci0 + ci)*kk + t]   for ci < Cin
  const int64_t total = (int64_t)Cout * kk * Cin;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int ci = (int)(i % Cin);
    const int t = (int)((i / Cin) % kk);
    const int co = (int)(i / ((int64_t)Cin * kk));
    const float v = w[((int64_t)co * cin_total + ci0 + ci) * kk + t] * wscale;   // power of two: exact
    const f16 hi = float_to_f16(v);
    // lo: the f16-rounded remainder of the split representation v ~= hi + lo (fp32-accurate mode)
    out[(int64_t)co * row_len + col_off + (int64_t)t * tap_width + ci] =
        lo ? float_to_f16(__fsub_rn(v, f16_to_float(hi))) : hi;
  }
}

// dgrad weights: the gradient of y = conv_{k x k, stride 1, pad k/2}(x, W) w.r.t. x is the same convolution of dy with
// W'[ci][co][t] = W[co][ci][kk-1-t]:  out[ci*row_len + col_off + t*tap_width + co] = w[(co*Cin + ci)*kk + (kk-1-t)]
__global__ void pack_weight_dgrad_kernel(const float* __restrict__ w, f16* __restrict__ out, int Cout, int Cin, int kk,
                                         int tap_width, int row_len, int col_off) {
  const int64_t total = (int64_t)Cout * kk * Cin;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int co = (int)(i % Cout);
    const int t = (int)((i / Cout) % kk);
    const int ci = (int)(i / ((int64_t)Cout * kk));
    out[(int64_t)ci * row_len + col_off + (int64_t)t * tap_width + co] =
        float_to_f16(w[((int64_t)co * Cin + ci) * kk + (kk - 1 - t)]);
  }
}

// fp32-accurate mode: the same weights times wscale (a power of two: exact), lo = 1 writes the f16-rounded remainder
// (the split representation v ~= hi + lo, as pack_weight_kernel)
__global__ void pack_weight_dgrad_split_kernel(const float* __restrict__ w, f16* __restrict__ out, int Cout, int Cin, int kk,
                                               int tap_width, int row_len, int col_off, int lo, float wscale) {
  const int64_t total = (int64_t)Cout * kk * Cin;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int co = (int)(i % Cout);
    const int t = (int)((i / Cout) % kk);
    const int ci = (int)(i / ((int64_t)Cout * kk));
    const float v = w[((int64_t)co * Cin + ci) * kk + (kk - 1 - t)] * wscale;
    const f16 hi = float_to_f16(v);
    out[(int64_t)ci * row_len + col_off + (int64_t)t * tap_width + co] = lo ? float_to_f16(__fsub_rn(v, f16_to_float(hi))) : hi;
  }
}

// dgrad of conv_in run as a 1x1 convolution over im2col columns: out[(t*Cin + ci)*row_len + co] = w[(co*Cin + ci)*9 + t]
__global__ void pack_weight_im2col_T_kernel(const float* __restrict__ w, f16* __restrict__ out, int Cout, int Cin, int row_len,
                                            int kk) {
  const int64_t total = (int64_t)Cout * Cin * kk;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int co = (int)(i % Cout);
    const int ci = (int)((i / Cout) % Cin);
    const int t = (int)(i / ((int64_t)Cout * Cin));
    out[(int64_t)(t * Cin + ci) * row_len + co] = float_to_f16(w[((int64_t)co * Cin + ci) * kk + t]);
  }
}

__global__ void pack_weight_im2col_T_split_kernel(const float* __restrict__ w, f16* __restrict__ out, int Cout, int Cin,
                                                  int row_len, int kk, int col_off, int lo, float wscale) {
  const int64_t total = (int64_t)Cout * Cin * kk;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int co = (int)(i % Cout);
    const int ci = (int)((i / Cout) % Cin);
    const int t = (int)(i / ((int64_t)Cout * Cin));
    const float v = w[((int64_t)co * Cin + ci) * kk + t] * wscale;
    const f16 hi = float_to_f16(v);
    out[(int64_t)(t * Cin + ci) * row_len + col_off + co] = lo ? float_to_f16(__fsub_rn(v, f16_to_float(hi))) : hi;
  }
}

__global__ void fill_identity_kernel(f16* __restrict__ out, int C, int row_len, int col_off, float value) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) out[(int64_t)c * row_len + col_off + c] = float_to_f16(value);
}

__global__ void pack_weight_up2_kernel(const float* __restrict__ w, f16* __restrict__ out, int Cout, int Cin, int tap_width,
                                       int row_len, int col_off, int phase, int lo, float wscale) {
  const int a = phase >> 1, b = phase & 1;
  const int64_t total = (int64_t)Cout * 4 * Cin;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int ci = (int)(i % Cin);
    const int t = (int)((i / Cin) % 4);
    const int co = (int)(i / ((int64_t)Cin * 4));
    const int th = t >> 1, tw = t & 1;
    // 3x3 rows / columns folded into this 2x2 tap
    const int kh0 = a == 0 ? (th == 0 ? 0 : 1) : (th == 0 ? 0 : 2), kh1 = a == 0 ? (th == 0 ? 0 : 2) : (th == 0 ? 1 : 2);
    const int kw0 = b == 0 ? (tw == 0 ? 0 : 1) : (tw == 0 ? 0 : 2), kw1 = b == 0 ? (tw == 0 ? 0 : 2) : (tw == 0 ? 1 : 2);
    const float* wp = w + ((int64_t)co * Cin + ci) * 9;
    float v = 0.f;
    for (int kh = kh0; kh <= kh1; ++kh)
      for (int kw = kw0; kw <= kw1; ++kw) v = __fadd_rn(v, wp[kh * 3 + kw]);
    v *= wscale;   // power of two: exact
    const f16 hi = float_to_f16(v);
    out[(int64_t)co * row_len + col_off + (int64_t)t * tap_width + ci] = lo ? float_to_f16(__fsub_rn(v, f16_to_float(hi))) : hi;
  }
}

int conv_pack_weight_up2(const float* w, f16* out, int Cout, int Cin, int tap_width, int row_len, int col_off, int phase,
                         cudaStream_t st, int lo, float wscale) {
  const int64_t total = (int64_t)Cout * 4 * Cin;
  int grid = (int)((total + 255) / 256);
  if (grid > kNumSMs * 16) grid = kNumSMs * 16;
  pack_weight_up2_kernel<<<grid, 256, 0, st>>>(w, out, Cout, Cin, tap_width, row_len, col_off, phase, lo, wscale);
  return check_launch("pack_weight_up2");
}

int conv_pack_weight(const float* w, f16* out, int Cout, int Cin, int ksize, int tap_width, int row_len,
                     int col_off, cudaStream_t st, int ci0, int cin_total, int lo, float wscale) {
  const int kk = ksize * ksize;
  const int64_t total = (int64_t)Cout * kk * Cin;
  int grid = (int)((total + 255) / 256);
  if (grid > kNumSMs * 16) grid = kNumSMs * 16;
  pack_weight_kernel<<<grid, 256, 0, st>>>(w, out, Cout, Cin, kk, tap_width, row_len, col_off, ci0,
                                           cin_total > 0 ? cin_total : Cin, lo, wscale);
  return check_launch("pack_weight");
}

int conv_pack_weight_dgrad(const float* w, f16* out, int Cout, int Cin, int ksize, int tap_width, int row_len, int col_off,
                           cudaStream_t st, int planes, float wscale) {
  const int kk = ksize * ksize;
  const int64_t total = (int64_t)Cout * kk * Cin;
  int grid = (int)((total + 255) / 256);
  if (grid > kNumSMs * 16) grid = kNumSMs * 16;
  if (planes == 3) {   // [W'_hi | W'_hi | W'_lo] x 2^10 per tap: taps 3 * tap_width apart, planes tap_width apart
    for (int k = 0; k < 3; ++k) {
      pack_weight_dgrad_split_kernel<<<grid, 256, 0, st>>>(w, out, Cout, Cin, kk, 3 * tap_width, row_len, col_off + k * tap_width,
                                                           k == 2, wscale);
      const int rc = check_launch("pack_weight_dgrad_split");
      if (rc) return rc;
    }
    return B2E_OK;
  }
  pack_weight_dgrad_kernel<<<grid, 256, 0, st>>>(w, out, Cout, Cin, kk, tap_width, row_len, col_off);
  return check_launch("pack_weight_dgrad");
}

int conv_pack_weight_im2col_T(const float* w, f16* out, int Cout, int Cin, int row_len, cudaStream_t st, int kk, int planes,
                              float wscale) {
  const int64_t total = (int64_t)Cout * Cin * kk;
  int grid = (int)((total + 255) / 256);
  if (grid > kNumSMs * 16) grid = kNumSMs * 16;
  if (planes == 3) {   // row_len = 3 * (columns per plane): [W_hi | W_hi | W_lo] x 2^10
    for (int k = 0; k < 3; ++k) {
      pack_weight_im2col_T_split_kernel<<<grid, 256, 0, st>>>(w, out, Cout, Cin, row_len, kk, k * (row_len / 3), k == 2,
                                                              wscale);
      const int rc = check_launch("pack_weight_im2col_T_split");
      if (rc) return rc;
    }
    return B2E_OK;
  }
  pack_weight_im2col_T_kernel<<<grid, 256, 0, st>>>(w, out, Cout, Cin, row_len, kk);
  return check_launch("pack_weight_im2col_T");
}

int conv_fill_identity(f16* out, int C, int row_len, int col_off, cudaStream_t st, float value) {
  fill_identity_kernel<<<(C + 255) / 256, 256, 0, st>>>(out, C, row_len, col_off, value);
  return check_launch("fill_identity");
}

// ------------------------------------------------------------------ host: TMA descriptors
static PFN_cuTensorMapEncodeTiled_v12000 get_encode() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (PFN_cuTensorMapEncodeTiled_v12000)p;
  }
  return fn;
}

static int encode_map(CUtensorMap* m, const void* ptr, int rank, const uint64_t* dims,
                      const uint64_t* strides_bytes, const uint32_t* box) {
  auto enc = get_encode();
  B2E_REQUIRE(enc, B2E_CUDA_ERROR, "cuTensorMapEncodeTiled entry point not available");
  uint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(m, B2E_TMA_DTYPE, (cuuint32_t)rank, const_cast<void*>(ptr),
                   (const cuuint64_t*)dims, (const cuuint64_t*)strides_bytes, (const cuuint32_t*)box,
                   (const cuuint32_t*)estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  B2E_REQUIRE(r == CUDA_SUCCESS, B2E_CUDA_ERROR,
              "cuTensorMapEncodeTiled failed (%d): rank %d dims [%llu %llu %llu %llu %llu] box [%u %u %u %u %u]",
              (int)r, rank, (unsigned long long)dims[0], (unsigned long long)dims[1],
              (unsigned long long)(rank > 2 ? dims[2] : 0), (unsigned long long)(rank > 3 ? dims[3] : 0),
              (unsigned long long)(rank > 4 ? dims[4] : 0), box[0], box[1], rank > 2 ? box[2] : 0,
              rank > 3 ? box[3] : 0, rank > 4 ? box[4] : 0);
  return B2E_OK;
}

int tma_encode_f16(CUtensorMap* m, const void* ptr, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                    const uint32_t* box) {
  return encode_map(m, ptr, rank, dims, strides_bytes, box);
}

static int pow2_divisor(int v, int cap) {
  int p = 1;
  while (p * 2 <= cap && v % (p * 2) == 0) p *= 2;
  return p;
}

int conv_cout_pad(int Cout) {
  if (Cout <= 16) return 16;
  if (Cout % 128 == 0) return Cout;
  return (Cout + 63) / 64 * 64;
}

// smallest number of 128 x 128 output tiles for which a 3x3 stride-1 layer runs on the halo kernels (B2E_HALO_MIN).
// Measured at batch 8 (profiles/README.md, r79) with the threshold lowered to 32 / 64: the 32x32 layers (128 tiles) gain
// 10-20 % over the plain SM-pair kernel, the 16x16 layers (64 tiles) are a wash against BN = 64 with twice the CTAs -
// +1 % on the step, inside run-to-run noise, so the default stays one full wave of SMs.
static int halo_min_tiles() {
  static const int v = getenv("B2E_HALO_MIN") ? atoi(getenv("B2E_HALO_MIN")) : kNumSMs;
  return v < 2 ? 2 : v;
}

ConvGeom conv_geometry(int N, int Ho, int Wo, int Cout, int ksize, int stride) {
  ConvGeom g;
  const int cout_pad = conv_cout_pad(Cout);
  g.Wt = pow2_divisor(Wo, kConvBlockM);
  g.Ht = pow2_divisor(Ho, kConvBlockM / g.Wt);
  g.Nt = kConvBlockM / (g.Wt * g.Ht);
  g.w_blks = Wo / g.Wt; g.h_blks = Ho / g.Ht; g.n_blks = (N + g.Nt - 1) / g.Nt;
  g.block_n = cout_pad <= 16 ? 16 : (cout_pad % 128 == 0 ? 128 : 64);
  // few output tiles (low-resolution levels): halve the N tile to double the number of CTAs - unless the layer can run
  // on the halo kernel, whose 3x lower L2 traffic per FLOP beats the extra CTAs
  const bool halo_shape = (ksize == 3 || ksize == 2) && stride == 1 && Wo % kHaloWt == 0 && Ho % kHaloHt == 0 && cout_pad % 128 == 0 &&
                          (int64_t)N * Ho * Wo / kConvBlockM * (cout_pad / 128) >= halo_min_tiles();
  static const int bn64_below = getenv("B2E_BN64_BELOW") ? atoi(getenv("B2E_BN64_BELOW")) : kNumSMs / 2;   // experiments
  if (g.block_n == 128 && !halo_shape && g.w_blks * g.h_blks * g.n_blks * (cout_pad / 128) < bn64_below) g.block_n = 64;
  // statistics are reduced over groups of block_n/8 rows, which must not straddle images
  g.stats_ok = g.block_n >= 64 && Cout % 64 == 0 && (g.Wt * g.Ht) % (g.block_n / 8) == 0;
  return g;
}

// (C, W, 1, H, N) view of an NHWC tensor (stride 1) or (2C, W/2, 2, H/2, N) (stride 2), box = one tile brick
// up2_phase >= 0: (N,H,W,C) is the sub-grid of pixels (2i + a, 2j + b) of a (N,2H,2W,C) tensor at `ptr`
static int encode_act_map(CUtensorMap* m, const f16* ptr, int N, int H, int W, int C, int stride,
                          int Wt, int Ht, int Nt, int pitch = 0, int halo_rows = 0, int up2_phase = -1) {
  const uint64_t e = 2;
  uint64_t dims[5], str[4];
  // halo_rows: extra rows of a halo brick (vertical taps - 1)
  uint32_t box[5] = {(uint32_t)kConvBlockK, (uint32_t)Wt, 1, (uint32_t)(Ht + halo_rows), (uint32_t)Nt};
  if (up2_phase >= 0) {
    const int a = up2_phase >> 1, b = up2_phase & 1;
    dims[0] = C; dims[1] = W; dims[2] = 1; dims[3] = H; dims[4] = N;
    str[0] = 2 * (uint64_t)C * e; str[1] = 2 * (uint64_t)(2 * W) * C * e; str[2] = str[1];
    str[3] = (uint64_t)(2 * H) * (2 * W) * C * e;
    return encode_map(m, ptr + ((int64_t)a * 2 * W + b) * C, 5, dims, str, box);
  }
  if (stride == 1) {
    const uint64_t P = pitch ? pitch : C;   // pixel pitch in elements (channel window of a wider tensor)
    dims[0] = C; dims[1] = W; dims[2] = 1; dims[3] = H; dims[4] = N;
    str[0] = P * e; str[1] = (uint64_t)W * P * e; str[2] = (uint64_t)W * P * e;
    str[3] = (uint64_t)H * W * P * e;
  } else {
    dims[0] = 2 * (uint64_t)C; dims[1] = W / 2; dims[2] = 2; dims[3] = H / 2; dims[4] = N;
    str[0] = 2 * (uint64_t)C * e; str[1] = (uint64_t)W * C * e; str[2] = 2 * (uint64_t)W * C * e;
    str[3] = (uint64_t)H * W * C * e;
  }
  return encode_map(m, ptr, 5, dims, str, box);
}

int conv_plan_build(ConvPlan* pl, const ConvDesc& d) {
  const int K = kConvBlockK;
  B2E_REQUIRE(d.s0.ptr && d.s0.C > 0 && d.s0.C % K == 0 && d.s1.C % K == 0 && d.r0.C % K == 0 && d.r1.C % K == 0,
              B2E_UNSUPPORTED_SHAPE, "conv: channel counts must be multiples of %d (got %d+%d, residual %d+%d)", K,
              d.s0.C, d.s1.C, d.r0.C, d.r1.C);
  B2E_REQUIRE(((d.ksize == 1 || d.ksize == 3) && d.up2_phase < 0 &&
               (d.stride == 1 || (d.stride == 2 && d.ksize == 3 && !d.s1.ptr && !d.r0.ptr))) ||
                  (d.up2_phase >= 0 && d.up2_phase < 4 && d.ksize == 2 && d.stride == 1 && !d.s1.ptr && !d.r0.ptr && !d.s0.pitch &&
                   !d.b_batch_rows && !d.gn_coef && d.out_f16),
              B2E_UNSUPPORTED_SHAPE, "conv: unsupported ksize/stride %d/%d", d.ksize, d.stride);
  B2E_REQUIRE(d.stride == 1 || (d.H % 2 == 0 && d.W % 2 == 0), B2E_UNSUPPORTED_SHAPE, "conv: stride 2 needs even H, W");
  B2E_REQUIRE(aligned16(d.s0.ptr) && (!d.s1.ptr || aligned16(d.s1.ptr)) && (!d.r0.ptr || aligned16(d.r0.ptr)) &&
                  (!d.r1.ptr || aligned16(d.r1.ptr)) && aligned16(d.w_packed) && (!d.out_f16 || aligned16(d.out_f16)),
              B2E_INVALID_ARG, "conv: unaligned tensor");
  B2E_REQUIRE(!d.r1.ptr || d.r0.ptr, B2E_INVALID_ARG, "conv: r1 without r0");
  B2E_REQUIRE(!d.out_f16 || d.Cout % 64 == 0, B2E_UNSUPPORTED_SHAPE,
              "conv: f16 NHWC output needs Cout %% 64 == 0 (got %d)", d.Cout);
  ConvPlan& p = *pl;
  p.N = d.N; p.Ho = d.H / d.stride; p.Wo = d.W / d.stride; p.Cout = d.Cout; p.cout_pad = conv_cout_pad(d.Cout);
  const ConvGeom g = conv_geometry(d.N, p.Ho, p.Wo, d.Cout, d.ksize, d.stride);
  p.Wt = g.Wt; p.Ht = g.Ht; p.Nt = g.Nt; p.w_blks = g.w_blks; p.h_blks = g.h_blks; p.n_blks = g.n_blks;
  p.block_n = g.block_n;
  // halo mode (p.halo = MT, the M tiles per CTA): big 3x3 stride-1 layers with 128-wide N tiles; a CTA owns an
  // (8*MT) x 16-pixel brick of one image, a cluster (SM pair) two bricks.  B2E_HALO=0 switches it off, =1 / =2
  // force MT.
  static const int halo_env = getenv("B2E_HALO") ? atoi(getenv("B2E_HALO")) : -1;
  p.halo = 0;
  p.up2_phase = d.up2_phase;
  if (halo_env != 0 && (d.ksize == 3 || d.up2_phase >= 0) && d.stride == 1 && (g.block_n == 128 || g.block_n == 16) && !d.b_batch_rows &&
      !d.s0.pitch && p.Wo % kHaloWt == 0 && p.Ho % kHaloHt == 0) {
    const int64_t tiles128 = (int64_t)d.N * p.Ho * p.Wo / kConvBlockM * (p.cout_pad / g.block_n);   // 128 x BN output tiles
    if (tiles128 >= halo_min_tiles() && tiles128 % 2 == 0) {
      p.halo = 1;
      // two M tiles per CTA share every B tile (10 KB instead of 14.7 KB from L2 per k-block, half the barrier
      // hand-shakes) but halve the number of work items: measured worth it from ~12 waves of SM pairs
      const bool mt2_ok = p.Ho % (2 * kHaloHt) == 0 && tiles128 % 4 == 0;
      if (mt2_ok && (halo_env == 2 || (halo_env < 0 && tiles128 / 4 >= 12 * (kNumSMs / 2)))) p.halo = 2;
    }
  }
  if (p.halo) {
    p.Wt = kHaloWt; p.Ht = kHaloHt; p.Nt = 1;
    p.w_blks = p.Wo / p.Wt; p.h_blks = p.Ho / p.Ht; p.n_blks = d.N;
  }
  B2E_REQUIRE(!d.tile_stats || (g.stats_ok && d.out_f16), B2E_UNSUPPORTED_SHAPE,
              "conv: fused GroupNorm statistics are not available for this output shape");
  B2E_REQUIRE(d.out_planes == 1 || (d.out_planes == 3 && d.out_f16 && !d.tile_stats), B2E_INVALID_ARG,
              "conv: split-f16 output needs 3 planes, an NHWC output and no fused statistics");
  p.split_pitch = d.out_planes == 3 ? d.Cout : 0;
  p.tile_stats = d.tile_stats;
  B2E_REQUIRE(!d.gn_coef || (d.stride == 1 && !d.b_batch_rows && !d.s0.pitch && d.out_planes == 1), B2E_UNSUPPORTED_SHAPE,
              "conv: the fused GroupNorm transform needs a stride-1 convolution with shared weights over plain f16 sources");
  p.gn_coef = d.gn_coef; p.gn_silu = d.gn_silu;
  p.coef_stride = d.s0.C + (d.s1.ptr ? d.s1.C : 0);
  p.taps = d.ksize * d.ksize;
  p.c0_chunks = d.s0.C / K;
  p.c1_chunks = d.s1.ptr ? d.s1.C / K : 0;
  p.r0_chunks = d.r0.ptr ? d.r0.C / K : 0;
  p.r1_chunks = d.r1.ptr ? d.r1.C / K : 0;
  for (int t = 0; t < p.taps; ++t) {
    const int kh = t / d.ksize, kw = t % d.ksize;
    if (d.up2_phase >= 0) {
      // phase (a, b): input rows {i + a - 1, i + a}, columns {j + b - 1, j + b} of the low-resolution tensor
      p.tap_dc[t] = 0; p.tap_dw[t] = (d.up2_phase & 1) - 1 + kw; p.tap_da[t] = 0; p.tap_dh[t] = (d.up2_phase >> 1) - 1 + kh;
    } else if (d.stride == 1) {
      p.tap_dc[t] = 0; p.tap_dw[t] = kw - d.ksize / 2; p.tap_da[t] = 0; p.tap_dh[t] = kh - d.ksize / 2;
    } else if (d.stride2_pad1) {
      // symmetric padding 1: input index 2*o + k - 1 -> (block o - 1, parity 1), (o, 0), (o, 1)
      p.tap_dc[t] = (kw != 1) * d.s0.C; p.tap_dw[t] = kw == 0 ? -1 : 0; p.tap_da[t] = kh != 1; p.tap_dh[t] = kh == 0 ? -1 : 0;
    } else {
      // diffusers Downsample2D with padding 0: pad (0,1,0,1), input index 2*o + k
      p.tap_dc[t] = (kw & 1) * d.s0.C; p.tap_dw[t] = kw >> 1; p.tap_da[t] = kh & 1; p.tap_dh[t] = kh >> 1;
    }
  }
  B2E_REQUIRE(d.stride == 1 || !d.s0.pitch, B2E_UNSUPPORTED_SHAPE, "conv: pitched input with stride 2");
  B2E_REQUIRE(!d.b_batch_rows || p.Nt == 1, B2E_UNSUPPORTED_SHAPE, "conv: batched B needs tiles within one image");
  // halo kernels: A boxes are the brick's halo (8*MT + 2 rows), residual boxes the brick (8*MT rows), the output
  // box one 8 x 16 M tile
  const int a_ht = p.halo ? p.Ht * p.halo : p.Ht;
  const int halo_rows = p.halo ? d.ksize - 1 : 0;     // 3x3: 2; sub-pixel phase (2x2): 1
  int rc = encode_act_map(&p.map_a0, d.s0.ptr, d.N, d.H, d.W, d.s0.C, d.stride, p.Wt, a_ht, p.Nt, d.s0.pitch, halo_rows);
  if (rc) return rc;
  p.map_a1 = p.map_a0; p.map_r0 = p.map_a0; p.map_r1 = p.map_a0; p.map_out = p.map_a0;
  if (d.s1.ptr && (rc = encode_act_map(&p.map_a1, d.s1.ptr, d.N, d.H, d.W, d.s1.C, d.stride, p.Wt, a_ht, p.Nt, 0, halo_rows))) return rc;
  if (d.r0.ptr && (rc = encode_act_map(&p.map_r0, d.r0.ptr, d.N, p.Ho, p.Wo, d.r0.C, 1, p.Wt, a_ht, p.Nt))) return rc;
  if (d.r1.ptr && (rc = encode_act_map(&p.map_r1, d.r1.ptr, d.N, p.Ho, p.Wo, d.r1.C, 1, p.Wt, a_ht, p.Nt))) return rc;
  p.has_out_f16 = d.out_f16 != nullptr;
  if (d.out_f16 && (rc = encode_act_map(&p.map_out, d.out_f16, d.N, p.Ho, p.Wo, d.Cout * d.out_planes, 1, p.Wt, p.Ht, p.Nt, 0, 0,
                                        d.up2_phase))) return rc;
  const uint64_t ktot = (uint64_t)p.taps * (d.s0.C + (d.s1.ptr ? d.s1.C : 0)) + (d.r0.ptr ? d.r0.C : 0) +
                        (d.r1.ptr ? d.r1.C : 0);
  uint64_t bd[2] = {ktot, d.b_batch_rows ? (uint64_t)d.N * d.b_batch_rows : (uint64_t)p.cout_pad};
  uint64_t bs[1] = {(d.b_pitch ? (uint64_t)d.b_pitch : ktot) * 2};
  p.b_batch_rows = d.b_batch_rows;
  // SM-pair mode: 128-wide N tiles, an even number of M tiles and enough tiles to keep every SM pair busy
  const int m_tiles = p.w_blks * p.h_blks * p.n_blks, tiles = m_tiles * (p.cout_pad / p.block_n);
  p.pair = (p.halo || (p.block_n == 128 && m_tiles % 2 == 0 && !d.b_batch_rows)) ? 1 : 0;
  // split-K when the tiles alone cannot fill the chip.  64-wide N tiles: the splits of a tile form a thread-block
  // cluster (up to 7 CTAs, at least 8 k-blocks each, all clusters co-resident) and exchange their partial accumulators
  // through distributed shared memory; other shapes: up to 8 splits of at least 8 k-blocks each through a global
  // fp32 workspace, finished by the CTA that arrives last.
  const int num_kb = (int)(ktot / K);
  p.splits = 1;
  p.split_cluster = 0;
  static const bool cluster_on = !(getenv("B2E_SPLIT_CLUSTER") && atoi(getenv("B2E_SPLIT_CLUSTER")) == 0);
  // (measured on B200 at batch 8: 28 -> 23 us on the 8x8 layers, +1 % on the whole step; B2E_SPLITK=0 disables)
  static const bool splitk_on = !(getenv("B2E_SPLITK") && atoi(getenv("B2E_SPLITK")) == 0);
  if (splitk_on && cluster_on && !p.pair && p.block_n == 64 && d.out_f16 && tiles * 2 <= kNumSMs) {
    int sp = kNumSMs / tiles;
    // more splits shorten the MMA phase but every extra partial tile costs 0.55 us of DSMEM ingress at the leader:
    // measured optimum (tools/conv_bench.py, B2E_SPLITK_MAX sweep) 3 splits at 36 k-blocks, 4 at 72, 5-7 at 144
    const int sp_k = num_kb >= 128 ? kConvMaxClusterSplits : num_kb >= 64 ? 4 : num_kb >= 24 ? 3 : num_kb / 8;
    if (sp > sp_k) sp = sp_k;
    if (sp > kConvMaxClusterSplits) sp = kConvMaxClusterSplits;
    static const int sp_max = getenv("B2E_SPLITK_MAX") ? atoi(getenv("B2E_SPLITK_MAX")) : kConvMaxClusterSplits;   // experiments
    if (sp > sp_max) sp = sp_max;
    while (sp >= 2 && conv_cluster_split_capacity(sp) < tiles) --sp;   // every cluster resident at once
    if (sp >= 2) { p.splits = sp; p.split_cluster = 1; }
  }
  if (p.splits == 1 && splitk_on && !p.pair && d.split_ws && d.out_f16 && tiles * 2 <= kNumSMs) {
    int sp = kNumSMs / tiles;
    if (sp > num_kb / 8) sp = num_kb / 8;
    static const int sp_max = getenv("B2E_SPLITK_MAX") ? atoi(getenv("B2E_SPLITK_MAX")) : kConvMaxSplits;   // experiments
    if (sp > kConvMaxSplits) sp = kConvMaxSplits;
    if (sp > sp_max) sp = sp_max;
    if (sp >= 2 && (size_t)tiles * sp * kConvBlockM * p.block_n * sizeof(float) <= d.split_ws_bytes) p.splits = sp;
  }
  p.split_ws = d.split_ws; p.split_counters = d.split_counters;
  uint32_t bb[2] = {(uint32_t)K, (uint32_t)(p.pair ? p.block_n / 2 : p.block_n)};
  rc = encode_map(&p.map_b, d.w_packed, 2, bd, bs, bb);
  if (rc) return rc;
  p.flops = 2.0 * d.N * p.Ho * p.Wo * (double)d.Cout * (double)ktot;
  return B2E_OK;
}

template <int BN, int STAGES, bool PAIR, bool HALO, int MT, int KPS, bool XF>
static int launch_x(const ConvPlan& pl, const ConvKParams& kp, int tiles, cudaStream_t st) {
  using Cfg = ConvCfg<BN, STAGES, PAIR, HALO, MT, KPS>;
  static_assert(Cfg::kSmemBytes <= 227 * 1024, "shared memory budget");
  static_assert(Cfg::kTmemCols <= 512, "TMEM budget");
  static bool attr_set = false;
  if (!attr_set) {
    B2E_CUDA(cudaFuncSetAttribute(conv_igemm_kernel<BN, STAGES, PAIR, HALO, MT, KPS, XF>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  Cfg::kSmemBytes));
    attr_set = true;
  }
  cudaLaunchConfig_t cfg = {};
  const int units = PAIR ? kNumSMs / 2 : kNumSMs;   // work items (tiles x splits, or tile pairs) in flight
  const int work = tiles * (PAIR ? 1 : kp.splits);
  cfg.gridDim = dim3((unsigned)((work < units ? work : units) * (PAIR ? 2 : 1)));
  if (!PAIR && kp.split_cluster) {
    // one work item per CTA, cluster = the splits of one tile (the plan guarantees work <= SMs and smem for the partials)
    B2E_REQUIRE(!HALO && work <= units && (size_t)(kp.splits - 1) * kConvBlockM * BN * sizeof(float) <= (size_t)Cfg::kRingBytes,
                B2E_INVALID_ARG, "conv: cluster split-K plan does not fit the kernel variant");
    cfg.gridDim = dim3((unsigned)work);
  }
  cfg.blockDim = dim3(XF ? kConvThreadsXf : kConvThreads);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = PAIR ? 2 : (kp.split_cluster ? kp.splits : 1); attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl_enabled() ? 2 : 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, conv_igemm_kernel<BN, STAGES, PAIR, HALO, MT, KPS, XF>, pl.map_a0, pl.map_a1, pl.map_r0,
                                     pl.map_r1, pl.map_b, pl.map_out, kp);
  if (e != cudaSuccess) { set_error("conv_igemm launch: %s", cudaGetErrorString(e)); return B2E_CUDA_ERROR; }
  return check_launch("conv_igemm");
}

// XF (fused GroupNorm of the A operand) is a second instantiation of every variant, selected per plan
template <int BN, int STAGES, bool PAIR, bool HALO = false, int MT = 1, int KPS = 1>
static int launch_t(const ConvPlan& pl, const ConvKParams& kp, int tiles, cudaStream_t st) {
  return kp.gn_coef ? launch_x<BN, STAGES, PAIR, HALO, MT, KPS, true>(pl, kp, tiles, st)
                    : launch_x<BN, STAGES, PAIR, HALO, MT, KPS, false>(pl, kp, tiles, st);
}

int conv_cluster_split_capacity(int splits) {
  static int cache[kConvMaxClusterSplits + 1] = {};
  if (splits < 2 || splits > kConvMaxClusterSplits) return 0;
  if (cache[splits]) return cache[splits] < 0 ? 0 : cache[splits];
  using Cfg = ConvCfg<64, 4, false, false, 1, 2>;
  auto kern = conv_igemm_kernel<64, 4, false, false, 1, 2, false>;
  int n = 0;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes) == cudaSuccess) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(splits * (kNumSMs / splits)));
    cfg.blockDim = dim3(kConvThreads);
    cfg.dynamicSmemBytes = Cfg::kSmemBytes;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = splits; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) { n = 0; cudaGetLastError(); }
  } else {
    cudaGetLastError();
  }
  cache[splits] = n > 0 ? n : -1;
  return n > 0 ? n : 0;
}

int conv_launch(const ConvPlan& pl, const ConvEpilogue& ep, cudaStream_t st) {
  B2E_REQUIRE(pl.has_out_f16 || ep.out_f32_nchw, B2E_INVALID_ARG, "conv: no output");
  B2E_REQUIRE(!(pl.has_out_f16 && pl.block_n == 16), B2E_UNSUPPORTED_SHAPE, "conv: f16 output with Cout <= 16");
  ConvKParams kp;
  kp.N = pl.N; kp.Ho = pl.Ho; kp.Wo = pl.Wo; kp.Cout = pl.Cout;
  kp.Wt = pl.Wt; kp.Ht = pl.Ht; kp.Nt = pl.Nt; kp.w_blks = pl.w_blks; kp.h_blks = pl.h_blks;
  kp.taps = pl.taps; kp.c0_chunks = pl.c0_chunks; kp.c1_chunks = pl.c1_chunks;
  kp.r0_chunks = pl.r0_chunks; kp.r1_chunks = pl.r1_chunks;
  for (int t = 0; t < 9; ++t) {
    kp.tap_dc[t] = pl.tap_dc[t]; kp.tap_dw[t] = pl.tap_dw[t]; kp.tap_da[t] = pl.tap_da[t]; kp.tap_dh[t] = pl.tap_dh[t];
  }
  kp.n_tiles = pl.cout_pad / pl.block_n;
  kp.b_batch_rows = pl.b_batch_rows;
  static const int dbg = getenv("B2E_DEBUG") ? atoi(getenv("B2E_DEBUG")) : 0;
  kp.debug = dbg;
  kp.splits = pl.splits; kp.split_ws = pl.split_ws; kp.split_counters = pl.split_counters;
  kp.split_cluster = pl.split_cluster;
  if (pl.up2_phase >= 0) { kp.halo_vt = 2; kp.halo_ht = 2; kp.halo_dh0 = (pl.up2_phase >> 1) - 1; kp.halo_dw0 = (pl.up2_phase & 1) - 1; }
  else { kp.halo_vt = 3; kp.halo_ht = 3; kp.halo_dh0 = -1; kp.halo_dw0 = -1; }
  kp.bias = ep.bias; kp.bias2 = ep.bias2; kp.temb = ep.temb; kp.temb_stride = ep.temb_stride;
  kp.out_f16 = pl.has_out_f16; kp.out_f32_nchw = pl.has_out_f16 ? nullptr : ep.out_f32_nchw;
  kp.tile_stats = pl.tile_stats;
  kp.split_pitch = pl.split_pitch;
  kp.relu = ep.relu;
  kp.acc_scale = ep.acc_scale;
  kp.gn_coef = reinterpret_cast<const float2*>(pl.gn_coef); kp.coef_stride = pl.coef_stride; kp.gn_silu = pl.gn_silu;
  kp.Hin = pl.Ho; kp.Win = pl.Wo;     // XF plans are stride-1 convolutions: input and output maps coincide
  // B2E_TRACE=<n>: the n-th halo launch (1-based) runs with clock64 tracing of CTA 0, then dumps to stderr
  kp.trace = nullptr;
  static const int trace_at = getenv("B2E_TRACE") ? atoi(getenv("B2E_TRACE")) : 0;
  static int halo_launches = 0;
  static long long* trace_buf = nullptr;
  const bool do_trace = trace_at > 0 && ++halo_launches == trace_at;
  if (do_trace) {
    if (!trace_buf) B2E_CUDA(cudaMalloc(&trace_buf, kTrAll * sizeof(long long)));
    B2E_CUDA(cudaMemsetAsync(trace_buf, 0, kTrAll * sizeof(long long), st));
    kp.trace = trace_buf;
  }
  struct TraceDump {
    bool on; cudaStream_t st; const long long* buf; const ConvPlan& pl;
    ~TraceDump() {
      if (!on) return;
      cudaStreamSynchronize(st);
      static long long h[kTrAll];
      cudaMemcpy(h, buf, sizeof(h), cudaMemcpyDeviceToHost);
      fprintf(stderr, "TRACE conv %dx%d taps %d chunks %d+%d res %d+%d pair %d\n", pl.Ho, pl.Wo, pl.taps, pl.c0_chunks,
              pl.c1_chunks, pl.r0_chunks, pl.r1_chunks, pl.pair);
      const long long t0 = h[kTrTotal - 1];
      fprintf(stderr, "KERNEL entry 0 roles_done %lld\n", h[kTrTotal - 2] - t0);
      long long g0 = 0;
      for (int b = 0; b < kTrCtaMax; ++b) if (h[kTrCta + 8 * b] && (!g0 || h[kTrCta + 8 * b] < g0)) g0 = h[kTrCta + 8 * b];
      for (int b = 0; b < kTrCtaMax && h[kTrCta + 8 * b]; ++b)
        fprintf(stderr, "CTA %d entry %lld ns, dependency resolved %lld, exit %lld, last-split reduce began %lld, chunks done %lld, store issued %lld, "
                "epilogue loop left %lld\n", b, h[kTrCta + 8 * b] - g0,
                h[kTrCta + 8 * b + 1] - g0, h[kTrCta + 8 * b + 2] - g0, h[kTrCta + 8 * b + 3] ? h[kTrCta + 8 * b + 3] - g0 : -1,
                h[kTrCta + 8 * b + 4] ? h[kTrCta + 8 * b + 4] - g0 : -1, h[kTrCta + 8 * b + 5] ? h[kTrCta + 8 * b + 5] - g0 : -1,
                h[kTrCta + 8 * b + 6] ? h[kTrCta + 8 * b + 6] - g0 : -1);
      for (int i = 0; i < 512 && h[kTrMma + i * 4 + 3]; ++i)
        fprintf(stderr, "MMA %d start %lld a_ready %lld b_ready %lld issued %lld\n", i, h[kTrMma + i * 4] - t0,
                h[kTrMma + i * 4 + 1] - t0, h[kTrMma + i * 4 + 2] - t0, h[kTrMma + i * 4 + 3] - t0);
      for (int i = 0; i < 256 && h[kTrPa + i * 3 + 2]; ++i)
        fprintf(stderr, "PA %d start %lld free %lld issued %lld\n", i, h[kTrPa + i * 3] - t0, h[kTrPa + i * 3 + 1] - t0,
                h[kTrPa + i * 3 + 2] - t0);
      for (int i = 0; i < 512 && h[kTrPb + i * 3 + 2]; ++i)
        fprintf(stderr, "PB %d start %lld free %lld issued %lld\n", i, h[kTrPb + i * 3] - t0, h[kTrPb + i * 3 + 1] - t0,
                h[kTrPb + i * 3 + 2] - t0);
      for (int i = 0; i < 64 && h[kTrEpi + i * 4 + 3]; ++i)
        fprintf(stderr, "EPI %d start %lld full %lld released %lld done %lld\n", i, h[kTrEpi + i * 4] - t0,
                h[kTrEpi + i * 4 + 1] - t0, h[kTrEpi + i * 4 + 2] - t0, h[kTrEpi + i * 4 + 3] - t0);
    }
  } trace_dump{do_trace, st, trace_buf, pl};
  const int grid = pl.w_blks * pl.h_blks * pl.n_blks * kp.n_tiles / (pl.halo ? pl.halo : 1);
  kp.num_tiles = pl.pair ? grid / 2 : grid;
  switch (pl.block_n) {
    case 16:   // conv_out (3-4 channels): bound by the A traffic, so the halo kernel's 3x reuse is what matters
      if (pl.halo == 2) return launch_t<16, 5, true, true, 2>(pl, kp, kp.num_tiles, st);   // 5 x (36 + 3) KB
      if (pl.halo == 1) return launch_t<16, 8, true, true, 1>(pl, kp, kp.num_tiles, st);   // 8 x (20 + 3) KB
      return launch_t<16, 5, false, false, 1, 2>(pl, kp, kp.num_tiles, st);                // 5 x 2 x 18 KB
    case 64: return launch_t<64, 4, false, false, 1, 2>(pl, kp, kp.num_tiles, st);   // 4 x 2 x 24 KB
    default:
      if (pl.halo == 2) return launch_t<128, 3, true, true, 2>(pl, kp, kp.num_tiles, st);   // 3 x (36 + 24) KB
      if (pl.halo == 1) return launch_t<128, 4, true, true, 1>(pl, kp, kp.num_tiles, st);   // 4 x (20 + 24) KB
      if (pl.pair)   // full grids are L2-bound: deep ring of single k-blocks; small grids are hand-shake-bound
        return kp.num_tiles >= kNumSMs / 2 ? launch_t<128, 7, true>(pl, kp, kp.num_tiles, st)                   // 7 x 24 KB
                                           : launch_t<128, 3, true, false, 1, 2>(pl, kp, kp.num_tiles, st);   // 3 x 2 x 24 KB
      return launch_t<128, 5, false>(pl, kp, kp.num_tiles, st);
  }
}

}  // namespace b2e

using namespace b2e;

extern "C" int b2e_act_dtype(void) { return kActIsBf16; }

// Test hook: y = conv(x) (+ residual) as f16 NHWC; residual (N,Ho,Wo,Cout) f16 or NULL exercises the
// identity residual segment.
extern "C" int b2e_conv2d_nhwc_f16(const void* x, const float* w, const float* bias, const void* residual, void* out,
                                    int64_t N, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int ksize, int stride,
                                    void* stream) {
  B2E_REQUIRE(x && w && out, B2E_INVALID_ARG, "conv2d: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int cout_pad = conv_cout_pad((int)Cout);
  const int kk = ksize * ksize;
  const int row_len = (int)(kk * Cin + (residual ? Cout : 0));
  const size_t wbytes = (size_t)cout_pad * row_len * sizeof(f16);
  f16* wp = nullptr;
  B2E_CUDA(cudaMalloc(&wp, wbytes));
  // split-K scratch so that small shapes exercise the split path exactly like inside the UNet
  const size_t split_bytes = (size_t)kNumSMs * kConvBlockM * 128 * sizeof(float);
  char* split_mem = nullptr;
  if (cudaMalloc(&split_mem, split_bytes + 4096) != cudaSuccess) { cudaFree(wp); set_error("conv2d: cudaMalloc failed"); return B2E_CUDA_ERROR; }
  cudaMemsetAsync(split_mem + split_bytes, 0, 4096, st);
  int rc = B2E_OK;
  do {
    if (cudaMemsetAsync(wp, 0, wbytes, st) != cudaSuccess) { set_error("conv2d: memset failed"); rc = B2E_CUDA_ERROR; break; }
    rc = conv_pack_weight(w, wp, (int)Cout, (int)Cin, ksize, (int)Cin, row_len, 0, st);
    if (rc) break;
    if (residual) {
      rc = conv_fill_identity(wp, (int)Cout, row_len, (int)(kk * Cin), st);
      if (rc) break;
    }
    ConvDesc d;
    d.s0 = ConvSrc{(const f16*)x, (int)Cin};
    if (residual) d.r0 = ConvSrc{(const f16*)residual, (int)Cout};
    d.N = (int)N; d.H = (int)H; d.W = (int)W; d.ksize = ksize; d.stride = stride;
    d.w_packed = wp; d.Cout = (int)Cout; d.out_f16 = (f16*)out;
    d.split_ws = (float*)split_mem; d.split_ws_bytes = split_bytes; d.split_counters = (int*)(split_mem + split_bytes);
    ConvPlan plan;
    rc = conv_plan_build(&plan, d);
    if (rc) break;
    ConvEpilogue ep;
    ep.bias = bias;
    rc = conv_launch(plan, ep, st);
  } while (0);
  cudaStreamSynchronize(st);
  cudaFree(wp);
  cudaFree(split_mem);
  return rc;
}

// Measurement hook: one convolution plan per weight copy (`copies` packed weight sets, so that consecutive launches
// miss the L2 like the layers of a network do), `iters` launches back to back on `stream`, CUDA-event time per launch.
// Inputs / weights are whatever the allocations hold (zero-filled): the kernel's timing does not depend on the values.
extern "C" int b2e_conv2d_bench_f16(int64_t N, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int ksize, int stride,
                                     int iters, int copies, float* us_per_launch, void* stream) {
  B2E_REQUIRE(us_per_launch && iters > 0 && copies > 0 && copies <= 256, B2E_INVALID_ARG, "conv2d_bench: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  const int cout_pad = conv_cout_pad((int)Cout);
  const int row_len = (int)(ksize * ksize * Cin);
  const size_t wbytes = ((size_t)cout_pad * row_len * sizeof(f16) + 1023) / 1024 * 1024;
  const size_t xbytes = (size_t)N * H * W * Cin * sizeof(f16);
  const size_t obytes = (size_t)N * (H / stride) * (W / stride) * cout_pad * sizeof(f16);
  const size_t split_bytes = (size_t)kNumSMs * kConvBlockM * 128 * sizeof(float);
  char *wp = nullptr, *xp = nullptr, *op = nullptr, *split_mem = nullptr;
  float* bias = nullptr;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  int rc = B2E_OK;
  do {
    if (cudaMalloc(&wp, wbytes * copies) != cudaSuccess || cudaMalloc(&xp, xbytes) != cudaSuccess ||
        cudaMalloc(&op, obytes) != cudaSuccess || cudaMalloc(&split_mem, split_bytes + 4096) != cudaSuccess ||
        cudaMalloc(&bias, sizeof(float) * cout_pad) != cudaSuccess) {
      set_error("conv2d_bench: cudaMalloc failed"); rc = B2E_CUDA_ERROR; break;
    }
    cudaMemsetAsync(wp, 0, wbytes * copies, st);
    cudaMemsetAsync(xp, 0, xbytes, st);
    cudaMemsetAsync(bias, 0, sizeof(float) * cout_pad, st);
    cudaMemsetAsync(split_mem + split_bytes, 0, 4096, st);
    std::vector<ConvPlan> plans(copies);
    for (int i = 0; i < copies && !rc; ++i) {
      ConvDesc d;
      d.s0 = ConvSrc{(const f16*)xp, (int)Cin};
      d.N = (int)N; d.H = (int)H; d.W = (int)W; d.ksize = ksize; d.stride = stride;
      d.w_packed = (const f16*)(wp + wbytes * i); d.Cout = cout_pad; d.out_f16 = (f16*)op;
      d.split_ws = (float*)split_mem; d.split_ws_bytes = split_bytes; d.split_counters = (int*)(split_mem + split_bytes);
      rc = conv_plan_build(&plans[i], d);
    }
    if (rc) break;
    ConvEpilogue ep;
    ep.bias = bias;
    for (int i = 0; i < copies && !rc; ++i) rc = conv_launch(plans[i], ep, st);   // warm-up
    if (rc) break;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaEventRecord(e0, st);
    for (int i = 0; i < iters && !rc; ++i) rc = conv_launch(plans[i % copies], ep, st);
    cudaEventRecord(e1, st);
    if (cudaStreamSynchronize(st) != cudaSuccess) { set_error("conv2d_bench: %s", cudaGetErrorString(cudaGetLastError())); rc = B2E_CUDA_ERROR; break; }
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    *us_per_launch = ms * 1000.f / iters;
  } while (0);
  if (e0) cudaEventDestroy(e0);
  if (e1) cudaEventDestroy(e1);
  cudaFree(wp); cudaFree(xp); cudaFree(op); cudaFree(split_mem); cudaFree(bias);
  return rc;
}

// Test hook: y = conv3x3(nearest_upsample_x2(x)) + bias computed as the four 2x2 sub-pixel phase convolutions over the
// low-resolution input (ConvDesc::up2_phase), f16 NHWC (N,H,W,Cin) -> (N,2H,2W,Cout).  Allocates temporaries and synchronises.
extern "C" int b2e_upsample_conv3x3_nhwc_f16(const void* x, const float* w, const float* bias, void* out, int64_t N, int64_t H,
                                             int64_t W, int64_t Cin, int64_t Cout, void* stream) {
  B2E_REQUIRE(x && w && out, B2E_INVALID_ARG, "upsample_conv3x3: null pointer");
  B2E_REQUIRE(Cin % kConvBlockK == 0 && Cout % 64 == 0, B2E_UNSUPPORTED_SHAPE, "upsample_conv3x3: Cin, Cout must be multiples of 64");
  cudaStream_t st = (cudaStream_t)stream;
  const int cout_pad = conv_cout_pad((int)Cout);
  const int row_len = (int)(4 * Cin);
  const size_t wbytes = (size_t)cout_pad * row_len * sizeof(f16);
  const size_t split_bytes = (size_t)kNumSMs * kConvBlockM * 128 * sizeof(float);
  char *wp = nullptr, *split_mem = nullptr;
  B2E_CUDA(cudaMalloc(&wp, 4 * wbytes));
  if (cudaMalloc(&split_mem, split_bytes + 4096) != cudaSuccess) { cudaFree(wp); set_error("upsample_conv3x3: cudaMalloc failed"); return B2E_CUDA_ERROR; }
  cudaMemsetAsync(wp, 0, 4 * wbytes, st);
  cudaMemsetAsync(split_mem + split_bytes, 0, 4096, st);
  int rc = B2E_OK;
  for (int ph = 0; ph < 4 && !rc; ++ph) {
    f16* wph = (f16*)(wp + ph * wbytes);
    rc = conv_pack_weight_up2(w, wph, (int)Cout, (int)Cin, (int)Cin, row_len, 0, ph, st);
    if (rc) break;
    ConvDesc d;
    d.s0 = ConvSrc{(const f16*)x, (int)Cin};
    d.N = (int)N; d.H = (int)H; d.W = (int)W; d.ksize = 2; d.stride = 1; d.up2_phase = ph;
    d.w_packed = wph; d.Cout = (int)Cout; d.out_f16 = (f16*)out;
    d.split_ws = (float*)split_mem; d.split_ws_bytes = split_bytes; d.split_counters = (int*)(split_mem + split_bytes);
    ConvPlan plan;
    rc = conv_plan_build(&plan, d);
    if (rc) break;
    ConvEpilogue ep;
    ep.bias = bias;
    rc = conv_launch(plan, ep, st);
  }
  cudaStreamSynchronize(st);
  cudaFree(wp);
  cudaFree(split_mem);
  return rc;
}
