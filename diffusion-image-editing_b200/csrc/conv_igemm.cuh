// Implicit-GEMM convolution on tcgen05 tensor cores (sm_100a): host-side plan + launcher.
#pragma once
#include "act_type.cuh"
#include "common.cuh"

namespace b2e {

constexpr int kConvBlockM = 128;  // output pixels per CTA tile (UMMA_M)
constexpr int kConvBlockK = 64;   // f16 channels per pipeline stage (one 128B swizzle row)

struct ConvSrc {
  const f16* ptr = nullptr;  // NHWC
  int C = 0;                  // channels used
  int pitch = 0;              // elements between consecutive pixels (0: = C); > C selects a channel window
};

// y = conv_{k x k, stride}(x0 ++ x1)  [+ W_r (r0 ++ r1)]  + bias (+ bias2) (+ temb[n, :])
// The optional second term is a 1x1 "residual segment" appended to the GEMM K dimension: with
// W_r = conv_shortcut weights it fuses the ResNet shortcut convolution, with W_r = I it is the plain
// residual add - either way the epilogue never touches the residual tensor.
struct ConvDesc {
  ConvSrc s0, s1;            // input (virtually concatenated along channels), (N,H,W,C)
  ConvSrc r0, r1;            // residual sources at OUTPUT resolution, (N,Ho,Wo,C); stride must be 1
  int N = 0, H = 0, W = 0;
  int ksize = 3, stride = 1; // stride 1: padding ksize/2; stride 2: ksize 3, padding (0,1,0,1) ...
  int stride2_pad1 = 0;      // ... or symmetric padding 1 (UNet2DModel downsample_padding = 1)
  const f16* w_packed = nullptr;  // f16 [cout_pad][row_len], row_len = k*k*(C0+C1) + Cr0 + Cr1
  // batched B operand (attention: Q K^T and P V): image n uses rows [n*b_batch_rows, +Cout) of a
  // [N*b_batch_rows][row_len] matrix whose rows are b_pitch elements apart (0: shared weights / dense rows)
  int b_batch_rows = 0, b_pitch = 0;
  int Cout = 0;
  f16* out_f16 = nullptr;  // NHWC (N,Ho,Wo,Cout) through TMA store; null -> fp32 NCHW output only
  // fp32-accurate mode: 3 -> the output is written as split f16, channel planes [hi | lo | hi] of Cout channels each
  // (pixel pitch 3*Cout): hi = f16(v), lo = f16(v - hi).  A consumer convolution reads it as ONE 3*Cout-channel
  // source against weights packed [W_hi | W_hi | W_lo], i.e. x_hi W_hi + x_lo W_hi + x_hi W_lo (error ~2^-17 relative)
  int out_planes = 1;
  // >= 0: one PHASE of "nearest-upsample x2 then 3x3 convolution" computed on the LOW-resolution input (N,H,W,C): output
  // pixels (2i + a, 2j + b), a = phase >> 1, b = phase & 1, only see two input rows {i + a - 1, i + a} and two columns
  // {j + b - 1, j + b}, so the 3x3 taps collapse into 2x2 taps with pre-summed weights (conv_pack_weight_up2): 2.25x fewer
  // FLOPs than convolving the upsampled tensor, which is never materialised.  ksize must be 2, stride 1; out_f16 is the
  // full (N,2H,2W,Cout) tensor, written through a strided tensor map.
  int up2_phase = -1;
  // optional fused GroupNorm statistics of the (f16-rounded) output: per (tile slot, channel) sum and
  // sum of squares, [conv_stats_slots()][Cout][2] floats; reduced per image by gn_finalize
  float* tile_stats = nullptr;
  // optional fused GroupNorm(+SiLU) of the input: the kernel normalises the A operand on the fly in shared memory,
  // y = f16(silu(x * scale + shift)) with (scale, shift) float2 [N][s0.C + s1.C] from gn_coeffs_launch - the
  // normalised activation tensor is never written to memory.  Stride 1 only.
  const float* gn_coef = nullptr; int gn_silu = 0;
  // optional split-K scratch shared by all layers of a model: fp32 partial tiles + per-tile arrival counters
  // (counters must be zero before the first launch; the kernel re-arms them)
  float* split_ws = nullptr; size_t split_ws_bytes = 0; int* split_counters = nullptr;
};

struct ConvEpilogue {
  const float* bias = nullptr;    // [Cout]
  const float* bias2 = nullptr;   // [Cout] (shortcut bias)
  const float* temb = nullptr;    // [N][temb_stride], already offset to this layer's columns
  int temb_stride = 0;
  float* out_f32_nchw = nullptr;  // NCHW [N,Cout,Ho,Wo] (network output)
  int relu = 0;                   // f16 NHWC output: max(v, 0) before the store
  // the accumulator is multiplied by acc_scale before bias / time embedding: 1 / wscale of weights packed with a
  // power-of-two scale (fp32-accurate mode: keeps the lo halves of the split weights out of the fp16 subnormals)
  float acc_scale = 1.f;
};

// Everything the kernel needs that is fixed per layer; built once at model-build time.
struct ConvPlan {
  CUtensorMap map_a0, map_a1, map_r0, map_r1, map_b, map_out;
  int N, Ho, Wo, Cout, cout_pad;
  int Wt, Ht, Nt, w_blks, h_blks, n_blks;
  int taps, c0_chunks, c1_chunks, r0_chunks, r1_chunks;
  int tap_dc[9], tap_dw[9], tap_da[9], tap_dh[9];
  int block_n;  // 16, 64 or 128
  int b_batch_rows;
  int splits; float* split_ws; int* split_counters;
  int split_cluster;   // 1: the splits of a tile run as one thread-block cluster and meet in the leader's smem (DSMEM)
  int halo;     // 0, or MT = M tiles per CTA of the halo kernel: (8*MT)x16-pixel bricks, one halo load serves 3 vertical taps
  int up2_phase;   // ConvDesc::up2_phase (halo kernels: 2 x 2 taps, halo offset (a - 1, b - 1))
  int pair;     // 1: SM-pair kernel (tcgen05.mma.cta_group::2, 256 x 128 tile per cluster)
  int has_out_f16;
  int split_pitch;   // channels per plane of a split-f16 output (0: plain f16)
  float* tile_stats;
  const float* gn_coef; int coef_stride; int gn_silu;   // fused GroupNorm transform of the A operand (null: none)
  double flops;
};

int conv_plan_build(ConvPlan* plan, const ConvDesc& d);
int conv_cout_pad(int Cout);
// Tile geometry of an (N,Ho,Wo,Cout) output and whether the epilogue can emit GroupNorm statistics for it.
struct ConvGeom { int Wt, Ht, Nt, w_blks, h_blks, n_blks, block_n, stats_ok; };
ConvGeom conv_geometry(int N, int Ho, int Wo, int Cout, int ksize = 1, int stride = 1);
inline int64_t conv_stats_slots(const ConvGeom& g) { return (int64_t)g.w_blks * g.h_blks * g.n_blks * g.Nt; }
int conv_launch(const ConvPlan& plan, const ConvEpilogue& ep, cudaStream_t st);

// 128B-swizzled f16 TMA descriptor (rank <= 5); shared by the tensor-core kernels
int tma_encode_f16(CUtensorMap* m, const void* ptr, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                    const uint32_t* box);

// Fused attention (csrc/flash_attn.cu): O = softmax(scale * Q K^T) V on head-major operands qh [NV][Tq][D],
// kh [NV][Tk][D], vht [NV][D][Tk] -> oh [NV][Tq][D]; D in {64, 128, 192}, Tq, Tk multiples of 128; keys >= valid_k masked
struct FlashPlan {
  CUtensorMap map_q, map_k, map_v;
  int NV, Tq, Tk, D;
  f16* out;
  double flops;
};
int flash_attn_plan_build(FlashPlan* pl, const f16* qh, const f16* kh, const f16* vht, f16* oh, int NV, int Tq, int Tk, int D);
// softmax_warps: 8 (two threads per query row) or 4 (one); the engine uses flash_attn_default_warps() (B2E_FLASH_WARPS)
int flash_attn_launch(const FlashPlan& pl, int valid_k, float scale, int softmax_warps, cudaStream_t st, int causal = 0);
int flash_attn_default_warps();

// fp32 [Cout][Cin][k][k] -> f16 out[co*row_len + col_off + t*tap_width + ci]   (t = kh*k + kw)
// (ci0, cin_total): pack only input channels [ci0, ci0 + Cin) of a weight with cin_total input channels
// lo = 1: pack the remainder f16(w - f16(w)) instead of f16(w) (split-f16 weights of the fp32-accurate mode)
// wscale: the weights are multiplied by this power of two first (the consumer's epilogue undoes it, ConvEpilogue::acc_scale)
// 2x2 taps of phase (a, b) of the upsample-then-3x3 convolution: tap (th, tw) = sum of the 3x3 taps it stands for
// (rows {0} | {1,2} for a = 0, {0,1} | {2} for a = 1; columns likewise with b), summed in fp32, then rounded / split
int conv_pack_weight_up2(const float* w, f16* out, int Cout, int Cin, int tap_width, int row_len, int col_off, int phase,
                         cudaStream_t st, int lo = 0, float wscale = 1.f);
int conv_pack_weight(const float* w, f16* out, int Cout, int Cin, int ksize, int tap_width, int row_len,
                     int col_off, cudaStream_t st, int ci0 = 0, int cin_total = 0, int lo = 0, float wscale = 1.f);
// dgrad weights (flipped taps, transposed channels): out[ci*row_len + col_off + t*tap_width + co] = w[(co*Cin+ci)*kk + kk-1-t]
int conv_pack_weight_dgrad(const float* w, f16* out, int Cout, int Cin, int ksize, int tap_width, int row_len, int col_off,
                           cudaStream_t st);
// dgrad of the im2col conv_in: out[(t*Cin + ci)*row_len + co] = w[(co*Cin + ci)*9 + t]
// (kk taps: 9 for the 3x3 conv_in, 49 for the 7x7 stem of the classifier network)
int conv_pack_weight_im2col_T(const float* w, f16* out, int Cout, int Cin, int row_len, cudaStream_t st, int kk = 9);
// out[c*row_len + col_off + c] = value for c < C (identity residual segment)
int conv_fill_identity(f16* out, int C, int row_len, int col_off, cudaStream_t st, float value = 1.f);

}  // namespace b2e
