/*
 * b200edit.h - C ABI of libb200edit.so: the B200 (sm_100a) guided denoising loop of
 * JohanLundberg12/diffusion-image-editing.
 *
 * The reference has no FFI layer of its own: its boundary for this path is the Python
 * module surface (src/diffusion_utils.py, ddim_inversion.py, ddpm_inversion.py,
 * attr_functions.py, mask_creator.py, Morphology.py, utils.py, transforms.py,
 * SegDiffEditPipeline.py).  Each entry point below replaces the body of the reference
 * function(s) cited beside it; the Python drop-in modules under
 * diffusion-image-editing_b200/ bind these symbols with ctypes (INTEGRATION.md).
 *
 * Conventions
 *  - every tensor argument is a DEVICE pointer to caller-owned, contiguous memory
 *    (fp32 NCHW unless stated); the library never allocates user-visible memory;
 *  - `stream` is a cudaStream_t passed as void*; all work is enqueued asynchronously;
 *  - every function returns 0 on success or a negative b2e_status; it never throws or
 *    exits.  b2e_last_error() returns a thread-local message for the last failure;
 *  - per-step scalar coefficients are formed on the host in fp32 with the reference's
 *    op order (b2e_step_coeffs_compute) and passed by value - no host sync in a step.
 */
#ifndef B200EDIT_H
#define B200EDIT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2E_VERSION 100

typedef enum {
  B2E_OK = 0,
  B2E_INVALID_ARG = -1,
  B2E_UNSUPPORTED_SHAPE = -2,
  B2E_WORKSPACE_TOO_SMALL = -3,
  B2E_CUDA_ERROR = -4,
  B2E_ARCH_MISMATCH = -5,
  B2E_NOT_FOUND = -6
} b2e_status;

int b2e_version(void);
const char* b2e_last_error(void);
/* 0 iff the current device is sm_100 (B200); B2E_ARCH_MISMATCH otherwise. */
int b2e_device_check(void);
/* Number of kernels this library has launched in this process (all threads). */
int64_t b2e_launch_count(void);

/* ------------------------------------------------------------------ step coefficients
 * src/diffusion_utils.py:6-24,76-81 (calculate_variance, compute_alpha_products,
 * get_previous_timestep) + the scalar part of DDIMScheduler.step / reverse_step
 * (src/ddpm_inversion.py:203-240).  All fp32, reference op order, no FMA contraction. */
typedef struct {
  float sqrt_a_t;     /* alphas_cumprod[t] ** 0.5                                   */
  float sqrt_b_t;     /* (1 - alphas_cumprod[t]) ** 0.5                             */
  float sqrt_a_prev;  /* alpha_prod_t_prev ** 0.5                                   */
  float dir_coef;     /* ddim: (1-a_prev-sigma**2)**0.5 ; ddpm: (1-a_prev-eta*var)**0.5 */
  float sigma;        /* eta * variance ** 0.5                                      */
  float a_t_sq;       /* alphas_cumprod[t] ** 2  (guidance step size, attr_functions.py:158) */
  float variance;
  float a_t;
  float a_prev;
} b2e_step_coeffs;

#define B2E_MODE_DDIM 0 /* DDIMScheduler.step  (single_step, src/diffusion_utils.py:90-109) */
#define B2E_MODE_DDPM 1 /* reverse_step        (src/ddpm_inversion.py:203-240)              */

/* alphas_cumprod: HOST pointer to the fp32 table (num_train entries). */
int b2e_step_coeffs_compute(const float* alphas_cumprod, int num_train, float final_alpha_cumprod,
                            int t, int t_prev, float eta, int mode, b2e_step_coeffs* out);

/* ------------------------------------------------------------------ fused guided step
 * One kernel for: x0 prediction (src/diffusion_utils.py:27-31) -> optional clip ->
 * DDIM / DDPM update (+ sigma*z) -> colour guidance of AttrFunc.apply with the analytic
 * gradient of single_color_loss / color_loss (src/attr_functions.py:22-37,104-163). */
typedef struct {
  b2e_step_coeffs c;
  int32_t clip;             /* scheduler.config.clip_sample (DDIM mode only)              */
  float clip_range;         /* scheduler.config.clip_sample_range                         */
  int32_t has_noise;        /* eta > 0: add c.sigma * z                                   */
  int32_t noise_batched;    /* z is (B,C,H,W) instead of the reference's (C,H,W)          */
  int32_t guide;            /* 0: no guidance (outside [t1,t2) or attr_func is None)      */
  int32_t has_target[4];    /* per channel: channel takes part in the colour loss          */
  float target[4];          /* tau_c                                                      */
  float coef[4];            /* k_c = loss_scale * w_c / N, formed on the host in fp32      */
  int32_t mask_grad;        /* mask_attr_grad: g <- mask * g                              */
  int32_t mask_batched;     /* mask is (B,C,H,W) instead of (1,C,H,W)                     */
  int32_t no_step;          /* x_t already is the post-step sample: guidance only
                               (AttrFunc.apply called on its own, attr_functions.py:120) */
} b2e_guided_step_params;

/* x_t, eps: (B,C,H,W); z: (C,H,W)|(B,C,H,W)|NULL; mask: (1|B,C,H,W)|NULL;
 * x_prev, x0_pred: (B,C,H,W) outputs (x0_pred may be NULL).  C <= 4. */
int b2e_guided_step_f32(const float* x_t, const float* eps, const float* z, const float* mask,
                        float* x_prev, float* x0_pred, int64_t B, int64_t C, int64_t HW,
                        const b2e_guided_step_params* p, void* stream);

/* Masked + L2-regularised guidance (calculate_loss, src/attr_functions.py:78-102 with
 * use_l2): loss = colour(mask*x0g) + lambda*||1 - mask*x0g - x_ref||_2.  Two passes over
 * the data (the norm is a global reduction).  workspace: b2e_l2reg_workspace_bytes(). */
typedef struct {
  b2e_guided_step_params base;
  float lambda_;
  float loss_scale;
} b2e_l2reg_params;
size_t b2e_l2reg_workspace_bytes(int64_t B, int64_t C, int64_t HW);
int b2e_guided_step_l2reg_f32(const float* x_t, const float* eps, const float* z, const float* mask,
                              const float* x_ref, float* x_prev, float* x0_pred, int64_t B, int64_t C,
                              int64_t HW, const b2e_l2reg_params* p, void* workspace,
                              size_t workspace_bytes, void* stream);

/* Guidance with an externally supplied gradient (user-defined AttrFunc.loss evaluated by
 * autograd in the host layer): x <- x + (mask? mask*g : g) * a_t_sq, g = -dL/dx given. */
int b2e_apply_guidance_grad_f32(float* x, const float* neg_grad, const float* mask, int64_t B,
                                int64_t CHW, int mask_batched, float a_t_sq, void* stream);

/* Analytic guidance THROUGH a latent decoder (LDM / SD; AttrFunc.apply with decode inside the graph,
 * src/attr_functions.py:120-163 + :22-37, :78-102): the built-in colour losses need no autograd - their gradient
 * w.r.t. the DECODED image is closed-form and enters b2e_vqdec_backward directly.
 *   d_img[b,c,p] = k[c] * sign(img - target[c])                      (0 where the channel has no target)
 * and, with use_mask_pred (mask_pred_original_sample + use_l2: loss(mask*img) + lambda*||1 - mask*img - x_0||_2):
 *   r = 1 - mask*img - x_ref ;  R = sqrt(sum_all r^2)  (one global reduction, fixed order, fp64 partials)
 *   d_img = mask * (k[c] * sign(mask*img - target[c]) - lam_scale * r / R)
 * k[c] = loss_scale * weight_c / N (N = B*H*W of the decoded image, or H*W per sample), lam_scale = loss_scale*lambda.
 * img, d_img (B,C,HW) fp32; mask (1|B,C,HW) or NULL; x_ref (B,C,HW) or NULL. */
typedef struct {
  int32_t has_target[4];
  float target[4];
  float k[4];
  float lam_scale;
  int32_t use_mask_pred;
  int32_t mask_batched;
} b2e_color_grad_params;
size_t b2e_color_loss_grad_workspace_bytes(void);
int b2e_color_loss_grad_f32(const float* img, const float* mask, const float* x_ref, float* d_img, int64_t B, int64_t C,
                            int64_t HW, const b2e_color_grad_params* p, void* workspace, size_t workspace_bytes,
                            void* stream);
/* The same colour gradient in the masked-prediction mode with the LPIPS regulariser instead of L2 (use_lpips):
 *   d_img = mask * k_c * sign(mask * img - target_c) + lam_scale * d_lpips
 * d_lpips = b2e_lpips_backward's d(LPIPS(1 - mask * img, x_0)) / d(img) (the -mask chain included); reads has_target,
 * target, k, lam_scale (= loss_scale * lambda_) and mask_batched of p; mask (1 | B, C, HW) is required. */
int b2e_lpips_guidance_grad_f32(const float* img, const float* mask, const float* d_lpips, float* d_img, int64_t B, int64_t C,
                                int64_t HW, const b2e_color_grad_params* p, void* stream);
/* ... and the update on the latent after the decoder's backward pass returned d_latent = dL/d(decoder input):
 *   g = -(d_latent * chain) / sqrt_a_t ;  x <- x + (mask? mask*g : g) * a_t_sq
 * chain = d(decoder input)/d(x0 prediction): 1 for LDM, 1/0.18215 for SD (src/diffusion_classes.py:33). */
int b2e_apply_latent_guidance_f32(float* x, const float* d_latent, const float* mask, int64_t B, int64_t CHW,
                                  int mask_batched, float chain, float sqrt_a_t, float a_t_sq, void* stream);

/* ------------------------------------------------------------------ single ops
 * compute_predicted_original_sample, src/diffusion_utils.py:27-31 */
int b2e_pred_x0_f32(const float* x_t, const float* eps, float* x0, int64_t n, float sqrt_a_t,
                    float sqrt_b_t, void* stream);
/* out = c_out_x0 * ((x - c_b*e) / c_a) + c_out_e * e : next_step (src/ddim_inversion.py:13-48)
 * and forward_step (src/ddpm_inversion.py:58-77). */
int b2e_renoise_f32(const float* x, const float* eps, float* out, int64_t n, float c_a, float c_b,
                    float c_out_x0, float c_out_e, void* stream);
/* get_noise_pred CFG combine, src/diffusion_utils.py:67-70: out = e0 + s*(e1 - e0) */
int b2e_cfg_combine_f32(const float* e_first, const float* e_second, float* out, int64_t n,
                        float scale, void* stream);
/* apply_mask, src/utils.py:23-28: out = mask*zv + (1-mask)*zo ; mask (1,C,H,W) broadcast over T */
int b2e_apply_mask_f32(const float* mask, const float* zo, const float* zv, float* out, int64_t T,
                       int64_t CHW, void* stream);
/* tensor_to_pil numerics, src/transforms.py:8-35: (B,C,H,W) fp32 -> (B,H,W,C) uint8,
 * u8 = trunc(clamp(x/2+0.5,0,1)*255) */
int b2e_to_uint8_f32(const float* x, uint8_t* out, int64_t B, int64_t C, int64_t HW, void* stream);

/* mu_tilde (src/ddpm_inversion.py:16-28) and other two-term blends: out = a*x + b*y */
int b2e_axpby_f32(const float* x, const float* y, float* out, int64_t n, float a, float b, void* stream);
/* Loss VALUES (the guidance update never needs them; kept for the reference's call surface).
 * l2_norm, src/attr_functions.py:11-13: out[0] = sqrt(sum (x-y)^2).
 * single_color_loss, src/attr_functions.py:22-25: out4[c] = mean_{b,h,w} |img[:,c] - targets4[c]|. */
size_t b2e_loss_workspace_bytes(void);
int b2e_l2_distance_f32(const float* x, const float* y, int64_t n, float* out, void* workspace,
                        size_t workspace_bytes, void* stream);
int b2e_channel_l1_f32(const float* img, int64_t B, int64_t C, int64_t HW, const float* targets4,
                       float* out4, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ loss heads of the network guidance
 * The part of NetAttrFunc / ClassifierAttrFunc that is not a dense network: loss value AND its analytic
 * gradient w.r.t. the network output (seed of the network's backward pass).
 * NetAttrFunc.loss, src/attr_functions.py:213-219: logits (C,HW) of batch element 0 (C <= 32);
 * p = softmax_c ; L = sum_{c in classes} sum_hw p[c] / area_divisor (the reference's literal 256*256);
 * dlogits[c,hw] = p[c,hw] * (1[c in classes] - sum_{k in classes} p[k,hw]) / area_divisor  (may be NULL).
 * classes: HOST int array of distinct ids.  loss: DEVICE fp32 [1]. */
size_t b2e_seg_area_head_workspace_bytes(void);
int b2e_seg_area_head_f32(const float* logits, int64_t C, int64_t HW, const int32_t* classes, int n_classes,
                          float area_divisor, float* loss, float* dlogits, void* workspace,
                          size_t workspace_bytes, void* stream);
/* ClassifierAttrFunc.loss, src/attr_functions.py:237-257: logits (n = B*80) viewed (-1,40,2); only batch row 0
 * is used: L = a[idx_for_class][idx_of_interest] (+ (a[reg_idx][reg_pred] + reg_score)^2 when reg_idx >= 0);
 * dlogits (n) = the matching one-hot(s), zero elsewhere (may be NULL; loss may be NULL). */
int b2e_classifier_head_f32(const float* logits, int64_t n, int idx_for_class, int idx_of_interest, int reg_idx,
                            int reg_pred, float reg_score, float* loss, float* dlogits, void* stream);
/* Per-sample heads (AttrFunc per_sample=True): the loss is sum_b L_b with L_b the head above on image b alone.
 * loss: DEVICE fp32 [B] (L_b); dlogits = dL_b/dlogits_b * grad_scale, the multiply being the last rounding step (the
 * rounding autograd applies when it seeds loss_scale into the head's backward; grad_scale 1 is exact).
 * Seg-area: logits (B,C,HW); the blocks and partial sums of one image depend on HW only, so image b's loss and gradient
 * bits are those of a B = 1 call on image b (b2e_seg_area_head_f32 IS the B = 1, grad_scale 1 case).
 * workspace: b2e_seg_area_head_batched_workspace_bytes(B). */
size_t b2e_seg_area_head_batched_workspace_bytes(int64_t B);
int b2e_seg_area_head_batched_f32(const float* logits, int64_t B, int64_t C, int64_t HW, const int32_t* classes,
                                  int n_classes, float area_divisor, float grad_scale, float* loss, float* dlogits,
                                  void* workspace, size_t workspace_bytes, void* stream);
/* Classifier: logits (B,80), one row per image; dlogits (B,80) holds every image's gradient row. */
int b2e_classifier_head_batched_f32(const float* logits, int64_t B, int idx_for_class, int idx_of_interest, int reg_idx,
                                    int reg_pred, float reg_score, float grad_scale, float* loss, float* dlogits,
                                    void* stream);

/* ------------------------------------------------------------------ edit-friendly inversion
 * sample_xts_from_x0, src/ddpm_inversion.py:31-55: xts[i] = x0*sa[i] + noise[i]*sb[i], i<T;
 * xts[T] = x0.  x0 (C,H,W); noise (T,C,H,W); sa, sb: DEVICE fp32 [T]; xts (T+1,C,H,W). */
int b2e_sample_xts_f32(const float* x0, const float* noise, const float* sa, const float* sb,
                       float* xts, int64_t T, int64_t CHW, void* stream);
/* z_t extraction, src/ddpm_inversion.py:135-169 (one step): mu = sqrt_a_prev*x0 + dir*eps;
 * z = (x_tm1 - mu)/sigma ; x_tm1 <- mu + sigma*z (in place).  Use mode DDPM coefficients. */
int b2e_extract_noise_f32(const float* x_t, const float* eps, float* x_tm1, float* z, int64_t n,
                          const b2e_step_coeffs* c, void* stream);

/* ------------------------------------------------------------------ masks
 * MaskCreator.create_mask (src/mask_creator.py:22-55) incl. Dilation2d(1,1,7,hard max)
 * (src/Morphology.py:47-111) and torchvision Resize (antialiased bilinear, ATen order).
 * seg: DEVICE int64 (H,W); classes: HOST int array; out: (1,channels,out_h,out_w) fp32 {0,1}. */
size_t b2e_mask_workspace_bytes(int64_t H, int64_t W, int64_t out_h, int64_t out_w);
int b2e_mask_from_seg(const int64_t* seg, int64_t H, int64_t W, const int32_t* classes,
                      int n_classes, int dilate, int ksize, int64_t out_h, int64_t out_w,
                      int channels, int antialias, float* out, void* workspace,
                      size_t workspace_bytes, void* stream);
/* N maps at once: seg DEVICE int64 (N,H,W) -> out (N,channels,out_h,out_w), the other arguments as b2e_mask_from_seg.
 * One launch per stage for the whole batch; map n comes out bit-identical to b2e_mask_from_seg on seg[n]. */
size_t b2e_mask_batched_workspace_bytes(int64_t N, int64_t H, int64_t W, int64_t out_h, int64_t out_w);
int b2e_mask_from_seg_batched(const int64_t* seg, int64_t N, int64_t H, int64_t W, const int32_t* classes,
                              int n_classes, int dilate, int ksize, int64_t out_h, int64_t out_w,
                              int channels, int antialias, float* out, void* workspace,
                              size_t workspace_bytes, void* stream);
/* Antialiased bilinear resize of one fp32 plane (H,W)->(out_h,out_w), ATen CPU order. */
int b2e_resize_bilinear_aa_f32(const float* in, int64_t H, int64_t W, float* out, int64_t out_h,
                               int64_t out_w, void* workspace, size_t workspace_bytes, void* stream);
/* Morphology.forward (src/Morphology.py:47-84): x (B,Cin,H,W), weight (Cout,Cin,k,k),
 * out (B,Cout,H,W); op 0 = dilation2d, 1 = erosion2d; soft_max with beta if soft != 0. */
int b2e_morphology2d_f32(const float* x, const float* weight, float* out, int64_t B, int64_t Cin,
                         int64_t Cout, int64_t H, int64_t W, int ksize, int op, int soft,
                         float beta, void* stream);

/* ------------------------------------------------------------------ UNet (noise predictor)
 * get_noise_pred's unconditional branch, src/diffusion_utils.py:72: eps = unet(x, t).sample
 * for a diffusers UNet2DModel (google/ddpm-celebahq-256 layout by default).  bf16 tensor-core
 * path: tcgen05 implicit-GEMM convolutions fed by TMA, fp32 accumulation in TMEM. */
typedef struct {
  int32_t sample_size;
  int32_t in_channels;
  int32_t out_channels;
  int32_t n_blocks;
  int32_t block_out_channels[8]; /* multiples of 8 and of norm_num_groups; non-multiples of 64 are zero-padded internally */
  int32_t down_attn[8]; /* 1: AttnDownBlock2D */
  int32_t up_attn[8];   /* 1: AttnUpBlock2D   */
  int32_t layers_per_block;
  int32_t norm_num_groups;
  float norm_eps;
  int32_t attention_head_dim; /* 0: single head */
  int32_t flip_sin_to_cos;
  float freq_shift;
  int32_t downsample_padding; /* 0: pad (0,1,0,1) before the stride-2 conv (DDPM-256); 1: symmetric padding 1 (LDM) */
  /* > 0: diffusers UNet2DConditionModel (Stable Diffusion 1.x layout): blocks flagged in down_attn / up_attn and the mid
   * block use Transformer2DModel (self-attention, cross-attention over the text tokens, GEGLU) instead of Attention */
  int32_t cross_attention_dim;
  int32_t num_attention_heads; /* SD 1.x: 8 (head_dim = channels / 8) */
  /* 0: bf16 operands (default).  1: fp32-accurate mode for the north star's 1e-4 bar (UNet2DModel only): activations and
   * weights are kept as split bf16 (hi + lo, ~16 mantissa bits) and every GEMM computes x_hi W_hi + x_lo W_hi + x_hi W_lo
   * on the same tcgen05 kernels with fp32 accumulation; GroupNorm / SiLU / softmax / attention run in fp32. */
  int32_t precision;
} b2e_unet_config;

typedef struct b2e_unet b2e_unet;

int b2e_unet_create(const b2e_unet_config* cfg, int64_t max_batch, b2e_unet** out);
void b2e_unet_destroy(b2e_unet* m);
/* Parameters by their diffusers state_dict names (for loading); fan_in = inputs per output unit
 * (PyTorch default-init bound 1/sqrt(fan_in)), 0 for normalisation scales / shifts. */
int b2e_unet_num_params(const b2e_unet* m);
int b2e_unet_param_info(const b2e_unet* m, int idx, const char** name, int64_t* numel, int64_t* fan_in);
/* Copy one fp32 parameter (DEVICE pointer, diffusers layout) into the model; it is repacked
 * to the kernel layout (bf16 [Cout][kh][kw][Cin] for convolutions) on `stream`. */
int b2e_unet_set_param(b2e_unet* m, const char* name, const float* data, int64_t numel, void* stream);
/* Activation arena: caller-owned device memory, bound once (TMA descriptors point into it). */
size_t b2e_unet_workspace_bytes(const b2e_unet* m);
int b2e_unet_bind_workspace(b2e_unet* m, void* workspace, size_t workspace_bytes);
/* x (B,Cin,S,S) fp32 NCHW; timesteps: DEVICE int64 [B]; eps (B,Cout,S,S) fp32 NCHW. */
int b2e_unet_forward(b2e_unet* m, const float* x, const int64_t* timesteps, float* eps, int64_t B,
                     void* stream);
double b2e_unet_flops(const b2e_unet* m, int64_t B);
/* Human-readable description of op `idx` of the current plan (shape, tiling); "" if out of range. */
/* get_noise_pred's CFG branch, src/diffusion_utils.py:61-70: eps = unet(x, t, encoder_hidden_states=context).sample for a
 * conditional UNet; context: DEVICE fp32 (B, ctx_len <= 128, cross_attention_dim) (the reference's (2,77,768) text_emb
 * for the doubled latent). */
int b2e_unet_forward_cond(b2e_unet* m, const float* x, const int64_t* timesteps, const float* context, int64_t ctx_len,
                          float* eps, int64_t B, void* stream);
const char* b2e_unet_op_desc(const b2e_unet* m, int idx);
/* One instrumented forward: CUDA events on `stream` around every op of the plan.  Per op: elapsed ms,
 * algorithmic FLOPs (convolutions / attention) or bytes (memory-bound ops) and kind
 * (0 tcgen05 convolution, 1 GroupNorm(+SiLU), 2 attention core, 3 other).  Synchronises the stream. */
int b2e_unet_profile(b2e_unet* m, const float* x, const int64_t* timesteps, float* eps, int64_t B,
                     void* stream, int max_ops, int* n_ops, float* ms, double* flops, double* bytes,
                     int* kind);
int b2e_unet_launches_per_forward(const b2e_unet* m);

/* ------------------------------------------------------------------ VQ decoder (LDM.decode)
 * src/diffusion_classes.py:62-70: vqvae.decode(latent.float()).sample for a diffusers VQModel
 * (CompVis/ldm-celebahq-256 `vqvae` layout by default): nearest-code quantisation -> post_quant_conv ->
 * Decoder (conv_in, mid block with single-head attention, up blocks, GroupNorm + SiLU, conv_out).
 * The handle is a b2e_unet*: parameters (diffusers state_dict names, e.g. "decoder.up_blocks.0.resnets.1.conv1.weight",
 * "quantize.embedding.weight", "post_quant_conv.weight"), workspace, forward (timesteps = NULL; x = latent
 * (B, latent_channels, S, S) fp32; output (B, out_channels, S << (n_blocks-1), ...) fp32) and profile use the
 * b2e_unet_* entry points. */
typedef struct {
  int32_t sample_size;       /* latent height = width */
  int32_t latent_channels;   /* 1, 3 or 4 */
  int32_t out_channels;
  int32_t n_blocks;
  int32_t block_out_channels[8]; /* bottom-up, as in the diffusers config: (128, 256, 512) */
  int32_t layers_per_block;
  int32_t norm_num_groups;
  float norm_eps;
  int32_t num_vq_embeddings; /* 0: no quantiser = AutoencoderKL.decode (post_quant_conv -> decoder), SD.decode */
  int32_t precision;         /* 0: bf16; 1: fp32-accurate (split-bf16 operands, forward only), as b2e_unet_config.precision */
} b2e_vqdec_config;
int b2e_vqdec_create(const b2e_vqdec_config* cfg, int64_t max_batch, b2e_unet** out);

/* ------------------------------------------------------------------ VQ / KL encoder (image -> latent)
 * LDM.encode (src/diffusion_classes.py:55-60): vqvae.encode(img).latents, and SD.encode (src/diffusion_classes.py:27-30):
 * vae.encode(img).latent_dist.mode() - the step before the path for real-image editing (prepare_for_edit,
 * src/SegDiffEditPipeline.py:95).  diffusers Encoder (conv_in -> DownEncoderBlock2D per level -> mid block with single-head
 * attention -> GroupNorm -> SiLU -> conv_out) + the 1x1 quant_conv, on the same engine as the UNet.  Parameters by their
 * diffusers names ("encoder.*", "quant_conv.*").  b2e_unet_forward(m, image, NULL, out, B, s): image (B, in_channels, S, S)
 * fp32 -> out (B, Q, S >> (n_blocks-1), ...) fp32 with Q = latent_channels (VQ: the pre-quantisation latents) or
 * 2 * latent_channels (double_z, KL: the moments [mean | logvar]; the distribution's mode is the first half). */
typedef struct {
  int32_t sample_size;       /* image height = width */
  int32_t in_channels;       /* 1, 3 or 4 */
  int32_t latent_channels;
  int32_t n_blocks;
  int32_t block_out_channels[8];
  int32_t layers_per_block;
  int32_t norm_num_groups;
  float norm_eps;
  int32_t double_z;          /* 1: AutoencoderKL (conv_out and quant_conv carry 2 * latent_channels) */
  /* 0: 16-bit operands; 1: fp32-accurate forward (split hi + lo operands, three products per GEMM, GroupNorm / SiLU /
   * attention in fp32), as b2e_vqdec_config.precision; the 1x1 quant_conv is fp32 either way */
  int32_t precision;
} b2e_vqenc_config;
int b2e_vqenc_create(const b2e_vqenc_config* cfg, int64_t max_batch, b2e_unet** out);
/* Gradient through the decoder (AttrFunc.apply with decode inside the graph, src/attr_functions.py:147-158):
 * b2e_unet_enable_grad(m, 1) switches the handle to gradient mode (every activation of a forward pass stays in the
 * workspace: re-query b2e_unet_workspace_bytes and re-bind); after b2e_unet_forward(m, latent, NULL, image, B, s),
 * b2e_vqdec_backward(m, d_image, d_latent, B, s) returns d(loss)/d(latent) (B, latent_channels, S, S) fp32 for
 * d(loss)/d(image) (B, out_channels, S_out, S_out) fp32.  The quantiser is straight-through (identity gradient), every
 * convolution gradient runs on the same tcgen05 kernel with flipped / transposed weights, bf16 gradients. */
int b2e_unet_enable_grad(b2e_unet* m, int enable);
int b2e_vqdec_backward(b2e_unet* m, const float* d_image, float* d_latent, int64_t B, void* stream);

/* ------------------------------------------------------------------ CLIP text encoder (prompt conditioning)
 * prep_text / encode_text, src/diffusion_utils.py:34-52: model.text_encoder(input_ids)[0] for the "" and prompt sequences,
 * i.e. transformers CLIPTextModel.last_hidden_state (token + position embedding, pre-LayerNorm transformer layers with
 * causal multi-head self-attention and a quick-GELU MLP, final LayerNorm).  Linear layers on the tcgen05 kernel (q/k/v fused
 * into one GEMM, residual adds as identity K segments), causal attention on the fused attention kernel (fp32-accurate
 * mode: on the causal tiled fp32 kernel, B2E_ATTN_FP32_TILED_CAUSAL).  Parameters by
 * their transformers names ("text_model.embeddings.token_embedding.weight", "text_model.encoder.layers.0.self_attn.q_proj.weight", ...).
 * b2e_clip_forward: input_ids DEVICE int64 (B, seq_len <= max_positions) -> hidden (B, seq_len, hidden_size) fp32.  The
 * tokenizer (BPE vocabulary files) stays the caller's. */
typedef struct {
  int32_t vocab_size;         /* 49408 */
  int32_t hidden_size;        /* 768 (SD 1.x: CLIP ViT-L/14 text tower) */
  int32_t intermediate_size;  /* 3072 */
  int32_t num_layers;         /* 12 */
  int32_t num_heads;          /* 12 */
  int32_t max_positions;      /* 77 */
  /* 0: 16-bit operands; 1: fp32-accurate forward (split hi + lo operands, three products per GEMM, embedding / LayerNorm /
   * quick-GELU in fp32, causal attention on the tiled fp32 kernel), as b2e_unet_config.precision */
  int32_t precision;
} b2e_clip_config;
int b2e_clip_create(const b2e_clip_config* cfg, int64_t max_batch, b2e_unet** out);
int b2e_clip_forward(b2e_unet* m, const int64_t* input_ids, int64_t seq_len, float* hidden, int64_t B, void* stream);

/* ------------------------------------------------------------------ classifier network (ClassifierAttrFunc)
 * The predictor of src/models.py:69-77 (torchvision resnet50 with an 80-way fc) inside ClassifierAttrFunc.loss,
 * src/attr_functions.py:237-257: logits = predictor(decode(x0)) and, through autograd in the reference, d(loss)/d(image).
 * torchvision ResNet (bottleneck or basic blocks) with eval-mode BatchNorm folded into the convolutions by the host:
 * parameters "conv1.weight/.bias", "layerL.B.convK.weight/.bias", "layerL.B.downsample.0.weight/.bias", "fc.weight/.bias".
 * 7x7 stem as an im2col GEMM, every convolution on the tcgen05 kernel with ReLU in the epilogue and the shortcut as a
 * fused K segment; b2e_unet_forward(m, image, NULL, logits, B, s): image (B, C, S, S) fp32 -> logits (B, num_classes);
 * b2e_resnet_backward: d(logits) (B, num_classes) fp32 -> d(image) (B, C, S, S) fp32 (dgrad twins of every convolution,
 * zero insertion for the stride-2 ones, max-pool / ReLU / pooling backward kernels).  Workspace, parameters and
 * profiling through the b2e_unet_* entry points. */
typedef struct {
  int32_t input_size;   /* image height = width: a power of two >= 64 */
  int32_t in_channels;  /* 1..4 */
  int32_t bottleneck;   /* 1: Bottleneck blocks (ResNet-50/101/152), 0: BasicBlock (ResNet-18/34) */
  int32_t layers[4];    /* (3, 4, 6, 3) for ResNet-50 */
  int32_t width;        /* 64 */
  int32_t num_classes;
  /* 0: classifier (global average pool + fc -> logits (B, num_classes)).
   * 1: face parser: BiSeNet (src/Segmentation/model.py:234-262, the network of SegmentationModel, src/models.py:80-118) on a
   *    basic-block backbone - context path with attention refinement, feature fusion, output head, bilinear
   *    (align_corners) upsampling: output = out[0] of the reference, logits (B, num_classes, S, S) fp32.  Created with
   *    gradient mode off (b2e_unet_enable_grad turns it on; b2e_resnet_backward then gives d(logits) -> d(image)).
   *    Parameters under the reference's names with BatchNorm folded ("cp.resnet.layer1.0.conv1.weight/.bias",
   *    "cp.arm16.conv.*", "cp.arm16.conv_atten.*", "cp.conv_head32.*", "cp.conv_avg.*", "ffm.convblk.*", "ffm.conv1.weight",
   *    "ffm.conv2.weight", "conv_out.conv.*", "conv_out.conv_out.*"). */
  int32_t head;
  /* 0: f16 operands throughout.  1 (head 0): fp32-accurate FORWARD - split f16 operands hi + lo, three tensor-core products
   * per GEMM, as b2e_unet_config.precision - so the ReLU / max-pool masks the backward pass reads agree with an fp32
   * evaluation of the network (a 16-bit forward flips the masks of near-zero activations, which dominates the error of
   * the INPUT GRADIENT); the backward pass stays on f16 operands unless grad_precision = 1. */
  int32_t precision;
  /* 0 (default): 16-bit backward - f16 gradients through f16 dgrad weights.  1 (needs precision = 1): fp32-accurate
   * backward - split gradients hi + lo through split dgrad weights [W'_hi | W'_hi | W'_lo] x 2^10 (three tensor-core
   * products per GEMM), every element-wise backward kernel in fp32.  The forward is the same either way.  Any other value,
   * or 1 with precision = 0: B2E_INVALID_ARG. */
  int32_t grad_precision;
} b2e_resnet_config;
int b2e_resnet_create(const b2e_resnet_config* cfg, int64_t max_batch, b2e_unet** out);
int b2e_resnet_backward(b2e_unet* m, const float* d_logits, float* d_image, int64_t B, void* stream);
/* Face parser (head 1) only: the forward of b2e_unet_forward, but the last op upsamples the head's logits and takes
 * their argmax per pixel in one kernel: labels DEVICE int64 (B, input_size, input_size) = torch.argmax(logits, 1) of the
 * logits b2e_unet_forward returns (first maximum on a tie, NaN counts as the maximum); no logits are written.  The pass
 * leaves no forward for b2e_resnet_backward.  B2E_INVALID_ARG on a classifier handle. */
int b2e_resnet_forward_labels(b2e_unet* m, const float* x, int64_t* labels, int64_t B, void* stream);

/* ------------------------------------------------------------------ LPIPS distance (use_lpips regulariser, metrics.lpips)
 * lpips v0.1 with net='vgg' (lpips.LPIPS(net='vgg'), normalize=False): scaling layer (x - shift) / scale, VGG-16
 * features[0:30] (thirteen 3x3 convolutions + ReLU, 2x2 max pools), taps relu1_2 .. relu5_3, per tap and pixel
 * sum_c w_k[c] (u0_c - u1_c)^2 of the channel-normalised features u = f / (||f|| + 1e-10), spatial mean, sum over taps.
 * Parameters under lpips.LPIPS().state_dict() names: "net.slice1.0.weight/.bias" .. "net.slice5.28.weight/.bias",
 * "lin0.model.1.weight" .. "lin4.model.1.weight" (the scaling layer's constants are built in).
 * b2e_lpips_set_reference: runs the network on x_ref (B_ref, 3, S, S) fp32 (B_ref = 1 or the batch of later forwards)
 *   and keeps its normalised tap features in a part of the workspace no forward overwrites.  Binding a workspace or
 *   toggling gradient mode drops the reference.
 * b2e_lpips_forward: dist[b] = LPIPS(mask ? 1 - mask * x : x, reference); x (B, 3, S, S) fp32, mask NULL or fp32
 *   (mask_batch = 1 or B, 3, S, S), dist (B) fp32.  Bit-deterministic (fixed-order fp64 reductions).
 * b2e_lpips_backward: d_x = d(sum_b d_dist[b] * dist[b]) / dx through the input transform of the last forward
 *   (b2e_lpips_forward of batch B; the gradient mode of b2e_unet_enable_grad is on after create).
 * Workspace, parameters and profiling through the b2e_unet_* entry points. */
typedef struct {
  int32_t input_size;   /* image height = width: a multiple of 16, >= 32 */
  int32_t precision;    /* 0: f16 operands; 1: fp32-accurate forward (backward on f16 operands unless grad_precision = 1),
                         * as b2e_resnet_config */
  int32_t grad_precision;   /* 0: 16-bit backward; 1 (needs precision = 1): fp32-accurate backward, as b2e_resnet_config */
} b2e_lpips_config;
int b2e_lpips_create(const b2e_lpips_config* cfg, int64_t max_batch, b2e_unet** out);
int b2e_lpips_set_reference(b2e_unet* m, const float* x_ref, int64_t B_ref, void* stream);
int b2e_lpips_forward(b2e_unet* m, const float* x, const float* mask, int64_t mask_batch, float* dist, int64_t B, void* stream);
int b2e_lpips_backward(b2e_unet* m, const float* d_dist, float* d_x, int64_t B, void* stream);

/* The 16-bit storage / tensor-core operand type the library was built for: 0 = IEEE fp16 (default), 1 = bf16
 * (-DB2E_ACT_BF16 builds).  Accumulation is fp32 either way. */
int b2e_act_dtype(void);

/* Test hook for the implicit-GEMM convolution: x (N,H,W,Cin) 16-bit NHWC (b2e_act_dtype), w (Cout,Cin,k,k) fp32,
 * bias fp32 [Cout] or NULL, residual (N,Ho,Wo,Cout) 16-bit NHWC or NULL (added through the fused
 * residual K-segment), out (N,Ho,Wo,Cout) 16-bit NHWC.  ksize 1|3, stride 1|2 (stride 2 pads
 * (0,1,0,1) like diffusers' Downsample2D).  Allocates temporaries itself and synchronises. */
int b2e_conv2d_nhwc_f16(const void* x, const float* w, const float* bias, const void* residual,
                         void* out, int64_t N, int64_t H, int64_t W, int64_t Cin, int64_t Cout,
                         int ksize, int stride, void* stream);

/* Test hook for the upsampler: out (N,2H,2W,Cout) = conv3x3(nearest_upsample_x2(x)) + bias, x (N,H,W,Cin) 16-bit NHWC,
 * w (Cout,Cin,3,3) fp32 - computed the way the engine does it (diffusers Upsample2D, src-side call: the UNets' and
 * decoders' `upsamplers.0`): four 2x2 sub-pixel phase convolutions over the LOW-resolution input with pre-summed weights,
 * each writing its sub-grid of the output through a strided TMA map.  Cin, Cout multiples of 64.  Allocates + synchronises. */
int b2e_upsample_conv3x3_nhwc_f16(const void* x, const float* w, const float* bias, void* out, int64_t N, int64_t H,
                                   int64_t W, int64_t Cin, int64_t Cout, void* stream);

/* Test hook for the attention kernels: out = softmax(Q K^T / sqrt(head_dim), keys < valid_k, causal) V per (image, head),
 * computed by the engine's own launch sequence of the named path (padding rules, shape checks, plans, launch order).
 * Operands are channel windows of 16-bit (b2e_act_dtype) token-major tensors, as the UNet hands them over:
 *   q   rows [B][H*W] of q_pitch channels, head h at channels q_col + h*head_dim;
 *   kv  rows [B][Tk] of kv_pitch channels, key head h at k_col + h*head_dim, value head h at v_col + h*head_dim;
 *   out rows [B][H*W] of out_pitch channels; the tail [heads*head_dim, out_pitch) is written with zeros.
 * The fp32 paths read and write split tensors of the fp32-accurate mode: every row is [hi | lo | hi] planes of `pitch`
 * channels each (value hi + lo); the pitches and columns above are then per plane.
 * The single-head, CUDA-core and fp32 split paths take one packed tensor (q == kv, q_pitch = kv_pitch = 3 * out_pitch,
 * columns 0 / out_pitch / 2 * out_pitch) and no key mask (Tk = H*W = valid_k).  causal (query i sees keys
 * <= min(i, valid_k - 1)) runs on the fused path and on B2E_ATTN_FP32_TILED_CAUSAL, which takes causal = 1 only (with
 * causal = 0 it is refused as an unknown path); softmax_warps (4 or 8) selects the fused kernel's softmax layout.  Every
 * unsupported combination returns an error before anything is launched.  Allocates temporaries itself and synchronises. */
enum {
  B2E_ATTN_FUSED = 0,         /* tcgen05 flash kernel (head_dim <= 192) between head gather / scatter */
  B2E_ATTN_MATERIALISED = 1,  /* batched Q K^T GEMM -> 16-bit scores -> masked row softmax -> P V GEMM */
  B2E_ATTN_SINGLE_HEAD = 2,   /* single-head GEMM attention straight from the qkv tensor */
  B2E_ATTN_CUDA_CORE = 3,     /* attention_kernel on the CUDA cores */
  B2E_ATTN_FP32_SPLIT = 4,    /* fp32-accurate attention_split_kernel */
  B2E_ATTN_FP32_TILED = 5,    /* fp32-accurate attention_split_tiled_kernel (online softmax over key tiles) */
  B2E_ATTN_FP32_TILED_CAUSAL = 6   /* its causal instantiation (key tiles above the diagonal skipped); causal = 1 */
};
int b2e_attention_f16(const void* q, int64_t q_pitch, int64_t q_col, const void* kv, int64_t kv_pitch, int64_t k_col,
                      int64_t v_col, void* out, int64_t out_pitch, int64_t B, int64_t H, int64_t W, int64_t Tk,
                      int64_t valid_k, int64_t heads, int64_t head_dim, int causal, int path, int softmax_warps,
                      void* stream);

/* Test hook for the backward of the fp32-accurate single-head self-attention O = softmax(Q K^T / sqrt(C)) V (the VQ / KL
 * decoders' mid-block attention in gradient mode): the flash-style fp32 kernels of the decoder backward alone.  All tensors
 * are split rows of the fp32-accurate mode, [hi | lo | hi] planes of `pitch` channels each (value hi + lo), b2e_act_dtype:
 *   qkv  (B, T, 9 * pitch): q | k | v blocks at columns 0 / pitch / 2 * pitch of every plane (C real channels each);
 *   o    (B, T, 3 * pitch): the forward output; d_o (B, T, 3 * pitch): d(loss)/dO;
 *   dq, dk, dv (B, T, 3 * pitch): the split gradients, tails [C, pitch) written with zeros.
 * T % 32 == 0, C % 8 == 0, 8 <= C <= 512.  Deterministic (no atomics).  Allocates its scratch itself and synchronises. */
int b2e_attention_bwd_fp32(const void* qkv, const void* o, const void* d_o, void* dq, void* dk, void* dv, int64_t B, int64_t T,
                           int64_t C, int64_t pitch, void* stream);

/* Test hook for the face parser's label kernel: x (N,Hi,Wi,planes*P) 16-bit NHWC (b2e_act_dtype; planes = 3: split
 * [hi | lo | hi] channel planes, value hi + lo) -> labels int64 (N,S,S), the argmax over the first K channels of the
 * align_corners bilinear upsampling to S x S. */
int b2e_bilinear_ac_argmax_f16(const void* x, int64_t* labels, int64_t N, int64_t Hi, int64_t Wi, int64_t P, int64_t K,
                               int64_t S, int planes, void* stream);

/* Measurement hook for the same kernel: `iters` back-to-back launches of one convolution (zero-filled operands of the
 * given shape, `copies` distinct packed weight sets used round-robin so that launches miss the L2 like the layers of a
 * network), CUDA-event time per launch in microseconds.  Allocates temporaries itself and synchronises. */
int b2e_conv2d_bench_f16(int64_t N, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int ksize, int stride,
                          int iters, int copies, float* us_per_launch, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200EDIT_H */
