// Memory-bound / small kernels around the tcgen05 convolutions of the UNet (f16 NHWC).
#pragma once
#include "conv_igemm.cuh"

namespace b2e {

// GroupNorm(+SiLU) over a (virtually concatenated) f16 NHWC tensor: statistics pass writes
// per-(image, chunk, group) partial sums; the apply pass reduces them (fixed order, fp64) and
// writes the normalised f16 tensor that the next convolution reads through TMA.
struct GNArgs {
  const f16* x0; const f16* x1;  // x1 may be null
  int C0, C1;      // REAL channels of each source (multiples of 8); groups are formed over the C0 + C1 real channels
  int P0, P1;      // channel pitch of each source (>= C; the tail [C, P) is zero padding and is skipped)
  int Pout;        // channel pitch of the output (>= C0 + C1): real channels are written compactly, the tail is zeroed
  int N, HW, G;
  float eps;
  const float* gamma; const float* beta;
  float* partial;  // [N][chunks][G][2]   (statistics pass; unused when cs0 is given)
  const float* cs0; const float* cs1;  // per-channel (sum, sumsq) of x0 / x1, [N][P][2], from the conv epilogue
  // small tensors: raw per-(tile slot, channel) statistics, reduced by gn_apply itself (no finalize launch)
  const float* ts0; const float* ts1;
  int ts_nt, ts_per_img;               // images per tile, tile slots per image (same geometry for both sources)
  int chunks;
  f16* out;       // [N][HW][Pout]
  int silu;
  float* save_stats = nullptr;   // optional [N][G][2] (mean, rstd) for the backward pass
  // 3: sources and output are split-f16 tensors of the fp32-accurate mode - channel planes [hi | lo | hi] of P
  // channels each (pixel pitch 3 * P), value = hi + lo; statistics must come from the stand-alone pass
  int planes = 1;
  int reverse = 0;   // apply pass walks the tensor back to front (L2 reuse of the producer's tail; set by gn_launch)
};

// Backward of y = GroupNorm(x) (optionally followed by SiLU), single source.  dx = d(loss)/dx (+ add):
//   xh = (x - mean) * rstd ; y = gamma * xh + beta ; dy = da * silu'(y) (or da) ; dxh = dy * gamma
//   dx = rstd * (dxh - mean_g(dxh) - xh * mean_g(dxh * xh))
// Two launches: per-(image, chunk, group) partial sums of (dxh, dxh * xh), then the apply pass.
struct GNBwdArgs {
  const f16* x;      // forward input, [N][HW][P] (C real channels)
  const f16* da;     // gradient w.r.t. the forward output, [N][HW][Pda]
  const f16* add;    // optional tensor added to dx (residual branch), [N][HW][P]
  f16* dx;           // [N][HW][P] (tail channels zeroed)
  int C, P, Pda;
  int N, HW, G;
  const float* gamma; const float* beta;
  const float* stats; // [N][G][2] (mean, rstd) saved by the forward
  float* partial;     // [N][chunks][G][2]
  int chunks;
  int silu;
};
int gn_bwd_launch(const GNBwdArgs& a, cudaStream_t st);
int gn_chunks(int HW, int C);
int gn_launch(const GNArgs& a, cudaStream_t st);
// fused GroupNorm: only the (scale, shift) coefficients, float2 [N][P0 + P1]; the consumer convolution applies them to its
// A operand in shared memory (ConvDesc::gn_coef) and the normalised tensor never exists in memory
int gn_coeffs_launch(const GNArgs& a, float* coef, cudaStream_t st);
// tile statistics written by the conv epilogue -> per-(image, channel) sums
int gn_finalize_launch(const float* tile_stats, float* chan_stats, int N, int C, int Nt, int w_blks, int h_blks,
                       cudaStream_t st, int phases = 1, int64_t phase_stride = 0);

// x fp32 NCHW (B,C,H,W) -> f16 NHWC (B,H,W,cpad), zero padded channels; im2col: channel t*C + c of a pixel holds
// x[c] at 3x3 tap t (zero outside the image), so that a 3x3 convolution becomes a 1x1 one
// planes = 3 (im2col only): split-f16 output [hi | lo | hi] of cpad channels each (fp32-accurate mode)
// gs (plain layout only): gradient scale record of grad_scale_launch, x is multiplied by gs[0]
// im2col only: mask (fp32 (1 | B, C, H, W), mask_batched) replaces x by 1 - mask * x, and shift / scale (C floats each,
// device) apply (v - shift[c]) / scale[c] (the LPIPS scaling layer) before the zero padding of the taps
int pack_input_launch(const float* x, f16* out, int B, int C, int H, int W, int cpad, bool im2col, cudaStream_t st,
                      int planes = 1, const float* gs = nullptr, const float* shift = nullptr, const float* scale = nullptr,
                      const float* mask = nullptr, int mask_batched = 0);
// gs[0] = s = 2^e, gs[1] = 1 / s with max|x| * mult * s in [4, 8) (B2E_GRAD_LOG2 moves the target); gs = 3 floats, gs[2] zero
// before the first launch (the kernels re-arm it).  Keeps fp16 gradients in range; exact (powers of two).
int grad_scale_launch(const float* x, int64_t n, float* gs, float mult, cudaStream_t st);
// nearest-neighbour x2 upsample, f16 NHWC
int upsample2x_launch(const f16* in, f16* out, int N, int H, int W, int C, cudaStream_t st);

// timestep embedding MLP and all per-resnet projections
struct TembArgs {
  const int64_t* timesteps;  // [B]
  int B, dim0, dim;          // dim0 = block_out[0], dim = 4*dim0
  int flip; float freq_shift;
  const float *w1, *b1, *w2, *b2;  // [dim][dim0], [dim], [dim][dim], [dim]
  const float *wp, *bp;            // [sumC][dim], [sumC]
  int sumC;
  float* act;   // [B][dim]   silu(temb)
  float* proj;  // [B][sumC]
};
int temb_launch(const TembArgs& a, cudaStream_t st);

// tensor-core attention pieces (single head, T >= 128): softmax over rows of S (f16 [rows][T], in place,
// logits scaled by `scale`) and V^T extraction qkv[N][T][3C] (v = columns [2C,3C)) -> vt[N][C][T]
int softmax_rows_launch(f16* s, int64_t rows, int T, float scale, cudaStream_t st);
int transpose_v_launch(const f16* qkv, f16* vt, int N, int T, int C, cudaStream_t st);

// transformer-block kernels (SD UNet2DConditionModel)
// (planes = 3: split-f16 rows of the fp32-accurate mode, [hi | lo | hi] planes per row)
int layernorm_rows_launch(const f16* x, f16* y, const float* gamma, const float* beta, int64_t rows, int C, float eps,
                          cudaStream_t st, int planes = 1);
int geglu_launch(const f16* in, f16* out, int64_t rows, int inner, cudaStream_t st, int planes = 1);
int pack_context_launch(const float* ctx, f16* out, int B, int L, int Lpad, int D, cudaStream_t st, int planes = 1);
int gather_heads_launch(const f16* src, f16* dst, int N, int Tsrc, int Tpad, int pitch, int col0, int heads, int d, int dpad,
                        bool transposed, cudaStream_t st);
int scatter_heads_launch(const f16* oh, f16* out, int N, int T, int Tpad, int pitch, int heads, int d, int dpad, cudaStream_t st);
int softmax_rows_masked_launch(f16* s, int64_t rows, int T, int valid, float scale, cudaStream_t st);

// CLIP text encoder helpers (planes = 3: split-f16 rows [hi | lo | hi] of D (quick_gelu: C) channels per plane; quick_gelu's
// numel then counts all three planes)
int clip_embed_launch(const int64_t* ids, const float* tok, const float* pos, f16* out, int B, int L, int Lpad, int D, int vocab,
                      cudaStream_t st, int planes = 1);
int quick_gelu_launch(const f16* in, f16* out, int64_t numel, cudaStream_t st, int planes = 1, int C = 0);
int unpad_rows_f32_launch(const f16* x, float* out, int B, int L, int Lpad, int D, cudaStream_t st, int planes = 1);

// backward helpers of the decoder (f16 NHWC gradients)
int downsum2x_launch(const f16* dy, f16* dx, int N, int H, int W, int C, cudaStream_t st);
int transpose_window_launch(const f16* src, f16* dst, int N, int R, int Cc, int src_pitch, int col0, cudaStream_t st);
int softmax_bwd_rows_launch(const f16* p, f16* dp, int64_t rows, int T, float scale, cudaStream_t st);
// mask (fp32 (1 | B, L, H, W), mask_batched): the chain of an input x -> 1 - mask * x, dz *= -mask
int vq_col2im_bwd_launch(const f16* dcols, const float* pq_w, float* dz, int B, int L, int H, int W, cudaStream_t st,
                         const float* gs = nullptr, const float* mask = nullptr, int mask_batched = 0);

// VQModel.decode front: nearest codebook entry + 1x1 post_quant_conv; z, out fp32 NCHW (B, L <= 4, HW)
int vq_quantize_launch(const float* z, const float* codebook, int n_codes, const float* pq_w, const float* pq_b, float* out,
                       int B, int L, int HW, cudaStream_t st);

// quant_conv of the VQ / KL encoders: out[n][o][p] = sum_c w[o][c] x[n][c][p] + b[o], fp32 NCHW, Cin, Cout <= 16
int pointwise_conv_f32_launch(const float* x, const float* w, const float* b, float* out, int B, int Cin, int Cout, int HW,
                              cudaStream_t st);

// classifier network (torchvision ResNet) kernels, csrc/resnet_kernels.cu
// planes = 3 / xplanes / yplanes = 3: split tensors [hi | lo | hi] of the fp32-accurate forward (pixel pitch 3 C)
int im2col7s2_launch(const float* x, f16* out, int B, int C, int H, int W, int KP, cudaStream_t st, int planes = 1);
int col2im7s2_launch(const f16* dcols, float* dx, int B, int C, int H, int W, int KP, cudaStream_t st, const float* gs = nullptr);
int maxpool3s2_launch(const f16* x, f16* y, uint8_t* idx, int N, int H, int W, int C, cudaStream_t st, int planes = 1);
int maxpool3s2_bwd_launch(const f16* x, const uint8_t* idx, const f16* gy, f16* gx, int N, int H, int W, int C, cudaStream_t st,
                          int xplanes = 1);
int relu_bwd_launch(const f16* g, const f16* y, f16* out, int64_t numel, cudaStream_t st, int yplanes = 1, int C = 0);
int subsample2x_launch(const f16* in, f16* out, int N, int Ho, int Wo, int C, cudaStream_t st);
int zero_upsample2x_launch(const f16* in, f16* out, int N, int Hi, int Wi, int C, cudaStream_t st);
int avgpool_fc_launch(const f16* x, float* feat, const float* w, const float* b, float* logits, int N, int HW, int C, int K,
                      cudaStream_t st, int planes = 1);
int avgpool_fc_bwd_launch(const float* dlogits, const float* w, float* dfeat, const f16* y, f16* g, int N, int HW, int C, int K,
                          cudaStream_t st, const float* gs = nullptr, int yplanes = 1);

// LPIPS (VGG-16) kernels, csrc/lpips_kernels.cu; planes / xplanes = 3: split tensors of the fp32-accurate forward
int maxpool2x2_launch(const f16* x, f16* y, uint16_t* idx, int N, int H, int W, int C, cudaStream_t st, int planes = 1);
int maxpool2x2_bwd_launch(const f16* x, const uint16_t* idx, const f16* gy, f16* gx, int N, int H, int W, int C, cudaStream_t st,
                          int xplanes = 1);
struct LpipsTaps { int n[5], off[5], hw[5]; };   // partial slots per tap, their offset in a row of partials, pixels per image
int lpips_head_blocks(int HW);
// mode 0: ref <- normalised features of x; mode 1: partial[b][slot0 ..] <- distance partial sums against ref
// hmax (mode 1): per-image running max of the head-gradient elements for d(dist) = 1 (zeroed by the caller per forward)
int lpips_head_launch(const f16* x, int B, int C, int HW, int planes, const float* w, float* ref, int ref_batched, double* partial,
                      int part_pitch, int slot0, int mode, float* hmax, cudaStream_t st);
// gs (grad_scale_launch record) from max_b |d_dist[b]| * hmax[b]; prod = B floats of scratch
int lpips_grad_scale_launch(const float* d_dist, const float* hmax, float* prod, int B, float* gs, cudaStream_t st);
int lpips_finalize_launch(const double* partial, int part_pitch, const LpipsTaps& taps, float* dist, int B, cudaStream_t st);
int lpips_head_bwd_launch(const f16* x, int B, int C, int HW, int planes, const float* w, const float* ref, int ref_batched,
                          const float* d_dist, const float* gs, const f16* gp, f16* gout, cudaStream_t st);

// face parser (BiSeNet) helpers
int avgpool_launch(const f16* x, float* feat, int N, int HW, int C, cudaStream_t st, int planes = 1);
int fc_act_launch(const float* x, const float* w, const float* b, float* out, int N, int C, int K, int act, cudaStream_t st);
int chan_affine_launch(const f16* x, const float* a, const float* b, const f16* y, f16* out, int N, int HW, int C,
                       cudaStream_t st, int planes = 1);
int bilinear_ac_launch(const f16* x, float* out, int N, int Hi, int Wi, int P, int K, int Ho, int Wo, cudaStream_t st, int planes = 1);
// the same upsampling, then the argmax over the K channels -> labels int64 (N,Ho,Wo)
int bilinear_ac_argmax_launch(const f16* x, int64_t* labels, int N, int Hi, int Wi, int P, int K, int Ho, int Wo, cudaStream_t st,
                              int planes = 1);
int bilinear_ac_bwd_launch(const float* g, f16* dx, int N, int Hi, int Wi, int P, int K, int Ho, int Wo, cudaStream_t st,
                           const float* gs = nullptr);
int chan_dot_launch(const f16* x, const f16* y, float* out, int N, int HW, int C, float scale, cudaStream_t st, int yplanes = 1);
int fc_t_launch(const float* g, const float* w, float* out, int N, int C, int K, float scale, cudaStream_t st);
int vec_act_bwd_launch(const float* g, const float* a, float* out, int n, int mode, cudaStream_t st);
int grad_merge_launch(const f16* g, const f16* e, int e_pitch, int e_off, const f16* y, f16* out, int64_t rows, int C,
                      cudaStream_t st, int yplanes = 1);

// multi-head tensor-core attention: head-major operands (virtual image v = n*heads + h, head_dim padded to 64)
int split_heads_launch(const f16* qkv, f16* qh, f16* kh, f16* vht, int N, int T, int P, int heads, int d, cudaStream_t st);
int merge_heads_launch(const f16* oh, f16* out, int N, int T, int P, int heads, int d, cudaStream_t st);

// single/multi-head self-attention core: qkv f16 [N][T][3P] (q | k | v blocks of P >= C channels) -> out f16 [N][T][P]
int attention_launch(const f16* qkv, f16* out, int N, int T, int C, int P, int heads, cudaStream_t st);
// fp32-accurate mode: qkv / out are split-f16 tensors ([hi | lo | hi] planes of 3P / P channels), arithmetic in fp32
int attention_split_launch(const f16* qkv, f16* out, int N, int T, int C, int P, int heads, cudaStream_t st);
// any sequence length (online softmax over key tiles); q / k / v are channel windows of split-f16 tensors with q_plane /
// k_plane channels per plane; keys >= valid_k are masked; out has o_plane channels per plane (o_real of them written).
// causal: query row r also sees no key past r (keys <= min(r, valid_k - 1)), a separate instantiation of the kernel
int attention_split_tiled_launch(const f16* q, int q_plane, int q_col, const f16* kv, int k_plane, int k_col, int v_col, f16* out,
                                 int o_plane, int o_real, int N, int Tq, int Tk_rows, int valid_k, int heads, int d, cudaStream_t st,
                                 int causal = 0);

}  // namespace b2e
