// Fused multi-head attention on the 5th-gen tensor cores (tcgen05, sm_100a): O = softmax(scale * Q K^T) V without ever
// writing the score matrix to HBM.
//
// Operands are the head-major, zero-padded copies the gather kernels produce ("virtual image" v = image * heads + head):
//   qh  [NV][Tq][D]   kh [NV][Tk][D]   vht [NV][D][Tk]  (= V^T)      D = head_dim padded to 64 / 128 / 192,
//   Tq, Tk multiples of 128; only the first `valid_k` keys take part (zero-padded text / 64-token maps).
// One persistent CTA per SM walks (v, 128-query block) work items.  Per item, two passes over the 128-key blocks:
//   pass A:  S = Q K^T (tcgen05.mma into TMEM)  ->  row maxima (every softmax thread owns one query row: no shuffles)
//   pass B:  S = Q K^T again -> P = exp2((S - max) * scale * log2 e) -> f16, 128B-swizzled smem tile (the A operand of
//            the second GEMM) -> O += P V (TMEM accumulator, never rescaled) ; row sums in registers
//   end:     O / rowsum -> f16 -> global.
// Recomputing Q K^T (1.5x the tensor work of the single-pass algorithm) buys an accumulator that never has to be
// rescaled, i.e. no TMEM read-modify-write on the critical path.  S is double-buffered in TMEM so the tensor cores
// compute block j+1's scores while the softmax warps work on block j.
// Warp roles: warp 0 = TMA producer (Q once per item; K (+ V^T) tiles through an smem ring), warp 1 = TMEM allocator +
// MMA issuer, warps 2-9 = softmax + epilogue (TMEM lane = query row; two threads per row, 64 key columns / half of the D
// output columns each, row maxima and sums exchanged through smem; softmax_warps = 4 selects one thread per row).
// Measured (r93): SD UNet forward at batch 16 30.45 -> 30.05 ms, LDM UNet at batch 32 14.74 -> 14.61 ms - the softmax
// warps were not the limiter the clock64 traces suggested; the remaining gap is in the MMA / TMEM hand-shakes.
#include <cudaTypedefs.h>
#include <stdlib.h>

#include "conv_igemm.cuh"
#include "tcgen05_ptx.cuh"

namespace b2e {

// 32 consecutive fp32 columns of this thread's TMEM lane; completion is awaited separately (tmem_ld_wait) so that the
// four loads of a 128-column score row are in flight together
__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,"
      "%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
// (tmem_ld_wait: tcgen05_ptx.cuh)

constexpr int kFaBlock = 128;   // queries per item and keys per block
// SW = softmax warps: 4 (one thread per query row, all 128 key columns) or 8 (two threads per row, 64 columns each: the
// softmax phase is issue- / MUFU-latency-bound with one warp per scheduler, two warps per scheduler hide it)
template <int SW> __device__ __forceinline__ void fa_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(32 * SW) : "memory"); }

template <int D>
struct FaCfg {
  static constexpr int kChunks = D / 64;                      // 64-channel K chunks of Q / K
  static constexpr int kQBytes = kChunks * kFaBlock * 128;    // Q tile: chunks x [128 rows][128 B]
  static constexpr int kKBytes = kQBytes;                     // K tile, same shape
  static constexpr int kVBytes = 2 * D * 128;                 // V^T tile: 2 key chunks x [D rows][128 B]
  static constexpr int kStages = D <= 128 ? 2 : 1;            // K/V ring (96 KB per stage at D = 192)
  static constexpr int kPBytes = 2 * kFaBlock * 128;          // P tile: 2 key chunks x [128 rows][128 B]
  static constexpr int kPBufs = 2;                            // double-buffered: softmax of block j+1 overlaps P V of block j
  static constexpr int kSmemBytes = kQBytes + kStages * (kKBytes + kVBytes) + kPBufs * kPBytes + 1024 + 256 + 1024;   // + row max / sum exchange [2][128] floats
  static constexpr int kTmemCols = 512;                       // S double buffer (2 x 128) + O (D <= 192)
  static constexpr uint32_t kSCol = 0, kOCol = 256;
};

struct FaParams {
  int NV, Tq, Tk, valid_k;
  int causal;          // 1: query i attends to keys <= i only (CLIP text encoder)
  float scale_log2e;   // softmax scale * log2(e)
  f16* out;           // [NV][Tq][D]
};

template <int D, int SW>
__global__ void __launch_bounds__(64 + 32 * SW, 1)
flash_attn_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                  const __grid_constant__ CUtensorMap map_v, const __grid_constant__ FaParams p) {
  using Cfg = FaCfg<D>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* q_s = smem;
  uint8_t* kv_s = q_s + Cfg::kQBytes;
  uint8_t* p_s = kv_s + Cfg::kStages * (Cfg::kKBytes + Cfg::kVBytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(p_s + Cfg::kPBufs * Cfg::kPBytes);
  uint64_t* kv_full = bars;                       // [kStages]
  uint64_t* kv_empty = kv_full + Cfg::kStages;    // [kStages]
  uint64_t* s_full = kv_empty + Cfg::kStages;     // [2]
  uint64_t* s_empty = s_full + 2;                 // [2]
  uint64_t* q_full = s_empty + 2;
  uint64_t* q_empty = q_full + 1;
  uint64_t* p_full = q_empty + 1;                 // [2]
  uint64_t* p_empty = p_full + 2;                 // [2]
  uint64_t* o_full = p_empty + 2;
  uint64_t* o_empty = o_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_empty + 1);
  float* xch = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 256);   // [2 halves][128 rows] max, then sum
  constexpr int H = SW / 4;            // column halves per query row
  constexpr int CW = kFaBlock / H;     // key columns per softmax thread and block

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int q_blocks = p.Tq / kFaBlock, n_kb = p.Tk / kFaBlock;
  const int num_items = p.NV * q_blocks;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&map_q); prefetch_tmap(&map_k); prefetch_tmap(&map_v);
    for (int s = 0; s < Cfg::kStages; ++s) { mbar_init(kv_full + s, 1); mbar_init(kv_empty + s, 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(s_full + s, 1); mbar_init(s_empty + s, SW); }
    mbar_init(q_full, 1); mbar_init(q_empty, 1);
    for (int s = 0; s < 2; ++s) { mbar_init(p_full + s, 1); mbar_init(p_empty + s, 1); }
    mbar_init(o_full, 1); mbar_init(o_empty, SW);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc<Cfg::kTmemCols>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();
  pdl_trigger();

  if (warp == 0) {
    // ===== TMA producer
    int stage = 0; uint32_t phase = 0;
    int it = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
      const int v = item / q_blocks, qb = item - v * q_blocks;
      mbar_wait(q_empty, (it & 1) ^ 1);   // the previous item's MMAs have finished reading Q
      if (elect_one()) {
        mbar_expect_tx(q_full, Cfg::kQBytes);
#pragma unroll
        for (int c = 0; c < Cfg::kChunks; ++c)
          tma_load_2d(q_s + c * (kFaBlock * 128), &map_q, q_full, c * 64, v * p.Tq + qb * kFaBlock);
      }
      __syncwarp();
      for (int pass = 0; pass < 2; ++pass) {
        for (int j = 0; j < n_kb; ++j) {
          mbar_wait(kv_empty + stage, phase ^ 1);
          uint8_t* ks = kv_s + stage * (Cfg::kKBytes + Cfg::kVBytes);
          if (elect_one()) {
            mbar_expect_tx(kv_full + stage, pass ? Cfg::kKBytes + Cfg::kVBytes : Cfg::kKBytes);
#pragma unroll
            for (int c = 0; c < Cfg::kChunks; ++c)
              tma_load_2d(ks + c * (kFaBlock * 128), &map_k, kv_full + stage, c * 64, v * p.Tk + j * kFaBlock);
            if (pass) {
#pragma unroll
              for (int kc = 0; kc < 2; ++kc)
                tma_load_2d(ks + Cfg::kKBytes + kc * (D * 128), &map_v, kv_full + stage, j * kFaBlock + kc * 64, v * D);
            }
          }
          __syncwarp();
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer
    constexpr uint32_t idesc_s = make_idesc(kFaBlock, kFaBlock);   // S = Q K^T : 128 x 128
    constexpr uint32_t idesc_o = make_idesc(kFaBlock, D);          // O += P V  : 128 x D
    int stage = 0; uint32_t phase = 0;
    uint32_t g = 0;      // running S-buffer counter (buffer = g & 1, use = g >> 1)
    uint32_t pj = 0;     // running P-tile counter
    int it = 0;
    auto issue_qk = [&](int st_, uint32_t gg) {
      const uint32_t b = gg & 1;
      mbar_wait(s_empty + b, ((gg >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t qa = smem_u32(q_s), ka = smem_u32(kv_s + st_ * (Cfg::kKBytes + Cfg::kVBytes));
      if (elect_one()) {
#pragma unroll
        for (int c = 0; c < Cfg::kChunks; ++c) {
          const uint64_t ad = make_smem_desc(qa + c * (kFaBlock * 128)), bd = make_smem_desc(ka + c * (kFaBlock * 128));
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_f16(tmem_base + Cfg::kSCol + b * kFaBlock, ad + (uint64_t)(k * 2), bd + (uint64_t)(k * 2), idesc_s,
                      (c > 0 || k > 0) ? 1u : 0u);
        }
        umma_commit(s_full + b);
      }
      __syncwarp();
    };
    for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
      mbar_wait(q_full, it & 1);
      tc_fence_after();
      // ---- pass A: scores only (row maxima)
      for (int j = 0; j < n_kb; ++j) {
        mbar_wait(kv_full + stage, phase);
        tc_fence_after();
        issue_qk(stage, g++);
        if (elect_one()) umma_commit(kv_empty + stage);   // K tile free once the scores are done
        __syncwarp();
        if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
      }
      // ---- pass B: scores -> (softmax warps) -> P V
      mbar_wait(o_empty, (it & 1) ^ 1);   // the previous item's epilogue has drained the O accumulator
      tc_fence_after();
      int st_j = stage; uint32_t ph_j = phase;   // stage of block j
      // scores of block 0
      mbar_wait(kv_full + st_j, ph_j);
      tc_fence_after();
      issue_qk(st_j, g++);
      for (int j = 0; j < n_kb; ++j) {
        int st_n = st_j + 1; uint32_t ph_n = ph_j;
        if (st_n == Cfg::kStages) { st_n = 0; ph_n ^= 1; }
        if (Cfg::kStages >= 2 && j + 1 < n_kb) {
          // scores of block j+1 while the softmax warps work on block j (needs its own K/V stage)
          mbar_wait(kv_full + st_n, ph_n);
          tc_fence_after();
          issue_qk(st_n, g++);
        }
        const uint32_t pb = pj & 1;
        mbar_wait(p_full + pb, (pj >> 1) & 1);
        tc_fence_after();
        const uint32_t pa = smem_u32(p_s + pb * Cfg::kPBytes), va = smem_u32(kv_s + st_j * (Cfg::kKBytes + Cfg::kVBytes) + Cfg::kKBytes);
        if (elect_one()) {
#pragma unroll
          for (int kc = 0; kc < 2; ++kc) {
            const uint64_t ad = make_smem_desc(pa + kc * (kFaBlock * 128)), bd = make_smem_desc(va + kc * (D * 128));
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_f16(tmem_base + Cfg::kOCol, ad + (uint64_t)(k * 2), bd + (uint64_t)(k * 2), idesc_o,
                        (j > 0 || kc > 0 || k > 0) ? 1u : 0u);
          }
          umma_commit(kv_empty + st_j);   // K and V^T of block j are free
          umma_commit(p_empty + pb);      // so is the P tile
          if (j == n_kb - 1) { umma_commit(o_full); umma_commit(q_empty); }
        }
        __syncwarp();
        ++pj;
        if (Cfg::kStages < 2 && j + 1 < n_kb) {
          // single-stage ring: block j+1's tiles can only arrive after block j's P V released the stage
          mbar_wait(kv_full + st_n, ph_n);
          tc_fence_after();
          issue_qk(st_n, g++);
        }
        st_j = st_n; ph_j = ph_n;
      }
      stage = st_j; phase = ph_j;
    }
  } else {
    // ===== softmax + epilogue: warp w owns TMEM lanes 32*(w%4) .. +31 ; thread = one query row
    const int q = warp & 3;              // TMEM lane quadrant this warp may read (warp id % 4)
    const int half = (warp - 2) >> 2;    // column half of the row this thread owns (always 0 with four softmax warps)
    const int r = q * 32 + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    uint32_t g = 0, pj = 0;
    int it = 0;
    for (int item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
      const int v = item / q_blocks, qb = item - v * q_blocks;
      // keys this query row may see: the valid prefix, cut at the diagonal for causal attention
      const int lim = p.causal ? min(p.valid_k, qb * kFaBlock + r + 1) : p.valid_k;
      // ---- pass A: row maximum over the valid keys
      float m = -INFINITY;
      for (int j = 0; j < n_kb; ++j, ++g) {
        const uint32_t b = g & 1;
        mbar_wait(s_full + b, (g >> 1) & 1);
        tc_fence_after();
        const int k0 = j * kFaBlock;
        uint32_t sr[CW / 32][32];
#pragma unroll
        for (int c = 0; c < CW / 32; ++c) tmem_ld32_nowait(lane_addr + Cfg::kSCol + b * kFaBlock + half * CW + c * 32, sr[c]);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(s_empty + b);   // the scores are in registers: hand the buffer back
        const int kc0 = k0 + half * CW;            // first key of this thread's columns
        if (kc0 + CW <= lim) {
#pragma unroll
          for (int c = 0; c < CW / 32; ++c)
#pragma unroll
            for (int e = 0; e < 32; ++e) m = fmaxf(m, __uint_as_float(sr[c][e]));
        } else {
#pragma unroll
          for (int c = 0; c < CW / 32; ++c)
#pragma unroll
            for (int e = 0; e < 32; ++e)
              if (kc0 + c * 32 + e < lim) m = fmaxf(m, __uint_as_float(sr[c][e]));
        }
      }
      if (H > 1) {   // the two threads of a row exchange their maxima
        xch[half * kFaBlock + r] = m;
        fa_bar_sync<SW>();
        m = fmaxf(xch[r], xch[kFaBlock + r]);
        fa_bar_sync<SW>();   // both values read before the buffer is reused for the row sums
      }
      const float mc = m * p.scale_log2e;
      // ---- pass B: probabilities -> P tile, row sum
      float l = 0.f;
      for (int j = 0; j < n_kb; ++j, ++g, ++pj) {
        const uint32_t b = g & 1;
        mbar_wait(s_full + b, (g >> 1) & 1);
        tc_fence_after();
        const int k0 = j * kFaBlock;
        uint32_t sr[CW / 32][32];
#pragma unroll
        for (int c = 0; c < CW / 32; ++c) tmem_ld32_nowait(lane_addr + Cfg::kSCol + b * kFaBlock + half * CW + c * 32, sr[c]);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(s_empty + b);   // the scores are in registers: hand the buffer back
        const uint32_t pb = pj & 1;
        mbar_wait(p_empty + pb, ((pj >> 1) & 1) ^ 1);   // the P V that last read this P buffer has finished
        uint8_t* ptile = p_s + pb * Cfg::kPBytes;
        const bool full_blk = k0 + half * CW + CW <= lim;
#pragma unroll
        for (int cl = 0; cl < CW / 16; ++cl) {   // 16 keys per step -> two 16-byte chunks of the row
          const int c = half * (CW / 16) + cl;     // 16-key step index within the 128-key block
          uint4 o0, o1;
          f16x2* ob0 = reinterpret_cast<f16x2*>(&o0);
          f16x2* ob1 = reinterpret_cast<f16x2*>(&o1);
          float pe[16];
#pragma unroll
          for (int e = 0; e < 16; ++e) {
            const float sc_ = __uint_as_float(sr[cl >> 1][(cl & 1) * 16 + e]);
            float v_;
            asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(v_) : "f"(fmaf(sc_, p.scale_log2e, -mc)));   // one MUFU op
            pe[e] = (full_blk || k0 + c * 16 + e < lim) ? v_ : 0.f;
          }
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            ob0[e] = floats_to_f16x2(pe[2 * e], pe[2 * e + 1]);
            ob1[e] = floats_to_f16x2(pe[8 + 2 * e], pe[8 + 2 * e + 1]);
          }
          // the row sum uses the ROUNDED probabilities: numerator (P V with f16 P) and denominator stay consistent
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 f0 = f16x2_to_float2(ob0[e]), f1 = f16x2_to_float2(ob1[e]);
            l += f0.x + f0.y + f1.x + f1.y;
          }
          // 128B-swizzled K-major tile: key chunk (c >> 2), row r, 16-byte chunk j stored at (j ^ (r & 7))
          uint8_t* row = ptile + (c >> 2) * (kFaBlock * 128) + r * 128;
          const int j0 = (c & 3) * 2;
          *reinterpret_cast<uint4*>(row + (((j0) ^ (r & 7)) << 4)) = o0;
          *reinterpret_cast<uint4*>(row + (((j0 + 1) ^ (r & 7)) << 4)) = o1;
        }
        fence_async_smem();   // generic-proxy smem writes -> visible to the tensor core (async proxy)
        fa_bar_sync<SW>();
        if (warp == 2 && lane == 0) mbar_arrive(p_full + pb);
      }
      if (H > 1) {   // the two threads of a row add their partial sums
        xch[half * kFaBlock + r] = l;
        fa_bar_sync<SW>();
        l = xch[r] + xch[kFaBlock + r];
        fa_bar_sync<SW>();
      }
      // ---- epilogue: O / l -> f16 -> global (the halves split the D columns)
      mbar_wait(o_full, it & 1);
      tc_fence_after();
      const float inv = 1.f / l;
      f16* orow = p.out + ((int64_t)v * p.Tq + qb * kFaBlock + r) * D;
#pragma unroll 1
      for (int c = half * (D / 16 / H); c < (half + 1) * (D / 16 / H); ++c) {
        float ov[16];
        tmem_ld16(lane_addr + Cfg::kOCol + c * 16, ov);
        uint4 o0, o1;
        f16x2* ob0 = reinterpret_cast<f16x2*>(&o0);
        f16x2* ob1 = reinterpret_cast<f16x2*>(&o1);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          ob0[e] = floats_to_f16x2(ov[2 * e] * inv, ov[2 * e + 1] * inv);
          ob1[e] = floats_to_f16x2(ov[8 + 2 * e] * inv, ov[8 + 2 * e + 1] * inv);
        }
        *reinterpret_cast<uint4*>(orow + c * 16) = o0;
        *reinterpret_cast<uint4*>(orow + c * 16 + 8) = o1;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(o_empty);
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<Cfg::kTmemCols>(tmem_base);
  }
}

template <int D, int SW>
static int flash_launch_t(const CUtensorMap& mq, const CUtensorMap& mk, const CUtensorMap& mv, const FaParams& p, cudaStream_t st) {
  using Cfg = FaCfg<D>;
  static_assert(Cfg::kSmemBytes <= 227 * 1024, "shared memory budget");
  static bool attr_set = false;
  if (!attr_set) {
    B2E_CUDA(cudaFuncSetAttribute(flash_attn_kernel<D, SW>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    attr_set = true;
  }
  const int items = p.NV * (p.Tq / kFaBlock);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(items < kNumSMs ? items : kNumSMs));
  cfg.blockDim = dim3(64 + 32 * SW);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl_enabled() ? 1 : 0;
  cudaError_t e = cudaLaunchKernelEx(&cfg, flash_attn_kernel<D, SW>, mq, mk, mv, p);
  if (e != cudaSuccess) { set_error("flash_attn launch: %s", cudaGetErrorString(e)); return B2E_CUDA_ERROR; }
  return check_launch("flash_attn");
}

int flash_attn_plan_build(FlashPlan* pl, const f16* qh, const f16* kh, const f16* vht, f16* oh, int NV, int Tq, int Tk, int D) {
  B2E_REQUIRE((D == 64 || D == 128 || D == 192) && Tq % kFaBlock == 0 && Tk % kFaBlock == 0 && NV >= 1, B2E_UNSUPPORTED_SHAPE,
              "flash_attn: unsupported shape NV %d Tq %d Tk %d D %d", NV, Tq, Tk, D);
  pl->NV = NV; pl->Tq = Tq; pl->Tk = Tk; pl->D = D; pl->out = oh;
  {
    uint64_t dims[2] = {(uint64_t)D, (uint64_t)NV * Tq}, str[1] = {(uint64_t)D * 2};
    uint32_t box[2] = {64, (uint32_t)kFaBlock};
    int rc = tma_encode_f16(&pl->map_q, qh, 2, dims, str, box);
    if (rc) return rc;
  }
  {
    uint64_t dims[2] = {(uint64_t)D, (uint64_t)NV * Tk}, str[1] = {(uint64_t)D * 2};
    uint32_t box[2] = {64, (uint32_t)kFaBlock};
    int rc = tma_encode_f16(&pl->map_k, kh, 2, dims, str, box);
    if (rc) return rc;
  }
  {
    uint64_t dims[2] = {(uint64_t)Tk, (uint64_t)NV * D}, str[1] = {(uint64_t)Tk * 2};
    uint32_t box[2] = {64, (uint32_t)D};
    int rc = tma_encode_f16(&pl->map_v, vht, 2, dims, str, box);
    if (rc) return rc;
  }
  pl->flops = 4.0 * NV * (double)Tq * Tk * D;
  return B2E_OK;
}

int flash_attn_default_warps() {
  // B2E_FLASH_WARPS=4: one softmax thread per query row (the original layout); default 8: two threads per row
  static const int sw = getenv("B2E_FLASH_WARPS") ? atoi(getenv("B2E_FLASH_WARPS")) : 8;
  return sw == 8 ? 8 : 4;
}

int flash_attn_launch(const FlashPlan& pl, int valid_k, float scale, int softmax_warps, cudaStream_t st, int causal) {
  B2E_REQUIRE(valid_k >= 1 && valid_k <= pl.Tk, B2E_INVALID_ARG, "flash_attn: valid_k %d of %d", valid_k, pl.Tk);
  B2E_REQUIRE(softmax_warps == 4 || softmax_warps == 8, B2E_INVALID_ARG, "flash_attn: %d softmax warps (4 or 8)", softmax_warps);
  FaParams p;
  p.NV = pl.NV; p.Tq = pl.Tq; p.Tk = pl.Tk; p.valid_k = valid_k; p.causal = causal; p.scale_log2e = scale * 1.4426950408889634f; p.out = pl.out;
  if (softmax_warps == 8) {
    switch (pl.D) {
      case 64: return flash_launch_t<64, 8>(pl.map_q, pl.map_k, pl.map_v, p, st);
      case 128: return flash_launch_t<128, 8>(pl.map_q, pl.map_k, pl.map_v, p, st);
      default: return flash_launch_t<192, 8>(pl.map_q, pl.map_k, pl.map_v, p, st);
    }
  }
  switch (pl.D) {
    case 64: return flash_launch_t<64, 4>(pl.map_q, pl.map_k, pl.map_v, p, st);
    case 128: return flash_launch_t<128, 4>(pl.map_q, pl.map_k, pl.map_v, p, st);
    default: return flash_launch_t<192, 4>(pl.map_q, pl.map_k, pl.map_v, p, st);
  }
}

}  // namespace b2e
