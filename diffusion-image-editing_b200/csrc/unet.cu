// UNet2DModel (diffusers layout) forward as a pre-planned sequence of sm_100a kernels.
//
// get_noise_pred's unconditional branch (src/diffusion_utils.py:72): eps = unet(x, t).sample.
// The model is described once as a small IR (resnet / attention / down / up nodes with the
// skip-connection stack resolved at build time), every convolution gets a ConvPlan (TMA
// descriptors + tile geometry) bound to fixed activation buffers in a caller-owned arena, and a
// forward pass is just the recorded list of launches on the caller's stream - no allocation,
// no host synchronisation, graph-capturable.
#include <math.h>
#include <string.h>

#include <functional>
#include <map>
#include <string>
#include <unordered_map>
#include <vector>

#include "attention.cuh"
#include "unet_kernels.cuh"

using namespace b2e;

namespace {

// res_c > 0: a 1x1 residual segment of res_c channels is appended to every weight row (shortcut / identity)
struct ConvL {
  f16* w = nullptr; float* b = nullptr; float* b2 = nullptr;
  int cin = 0, cin_pad = 0, cout = 0, cout_pad = 0, k = 0, res_c = 0, row_len = 0;
  int dg = -1;   // decoder: index of the dgrad twin (flipped / transposed weights) in b2e_unet::dgrads
  // upsampler convolutions: the four sub-pixel phases' 2x2-tap weights, [4][cout_pad][row_len_up2] (conv_pack_weight_up2)
  f16* w_up2 = nullptr; int row_len_up2 = 0;
};
struct NormL { float* g = nullptr; float* b = nullptr; int C = 0; };
struct ResnetL {
  std::string name; int cin0 = 0, cin1 = 0, cout = 0; NormL n1, n2; ConvL c1, c2, sc; bool has_sc = false;
  int temb_off = 0;
  int sc_dg = -1;   // decoder: dgrad twin of the 1x1 shortcut convolution
};
struct AttnL { std::string name; int C = 0, P = 0; NormL gn; ConvL qkv, proj; int qkv_dg = -1; };   // P = pad64(C): q | k | v blocks of P columns

// Channel counts that are not multiples of 64 (LDM: 224, 672) live in tensors whose channel pitch is rounded up to
// the 64-channel K chunk of the convolution kernel; the tail channels are identically zero (zero weight rows,
// biases and time-embedding columns produce them, zero weight columns ignore them).  Only GroupNorm and the
// attention core need the real count.
inline int pad64(int c) { return (c + 63) / 64 * 64; }

// Transformer2DModel of the SD UNet2DConditionModel: GroupNorm -> 1x1 proj_in -> BasicTransformerBlock (LayerNorm +
// self-attention, LayerNorm + cross-attention over the text tokens, LayerNorm + GEGLU feed-forward, each with its
// residual fused into the output projection's K segment) -> 1x1 proj_out + block input
struct LNL { float* g = nullptr; float* b = nullptr; int C = 0; };
struct XfL {
  std::string name; int C = 0, heads = 0, d = 0;
  NormL gn; LNL ln1, ln2, ln3;
  ConvL proj_in, qkv1, out1, q2, kv2, out2, ff1, ff2, proj_out;
};

enum NodeKind { N_RESNET, N_ATTN, N_DOWN, N_UP, N_PUSH, N_POPCAT, N_XFORMER };
struct Node { NodeKind kind; int idx; };

struct Tensor {
  f16* p = nullptr; int N = 0, H = 0, W = 0, C = 0; size_t bytes = 0;   // C = channel pitch (multiple of 64 for conv operands)
  int Cr = 0;               // real channels (<= C)
  float* cstats = nullptr;  // per-(image, channel) sum / sum of squares from the producing conv's epilogue
  float* tstats = nullptr;  // small tensors: raw per-(tile slot, channel) statistics instead (no finalize kernel)
  size_t tstats_bytes = 0; int ts_nt = 0, ts_per_img = 0;
  // fused GroupNorm: this "tensor" is the normalised VIEW of raw source(s) - p (C0 channels) ++ p1 (C1 channels) - that the
  // consumer convolution materialises on the fly in shared memory from gn_coef (float2 [N][C0 + C1]); it owns no memory
  bool alias = false; f16* p1 = nullptr; int C0 = 0, C1 = 0; float* gn_coef = nullptr; int gn_silu = 0;
};

struct Arena {
  char* base = nullptr; size_t cap = 0, off = 0, peak = 0;
  std::multimap<size_t, char*> free_list;
  bool dry = true;
  void reset(void* b, size_t c) {
    dry = (b == nullptr);
    base = dry ? (char*)(uintptr_t)(1 << 20) : (char*)b;  // dry run: fake, unique, non-null addresses
    cap = c; off = 0; peak = 0; free_list.clear();
  }
  void* alloc(size_t n) {
    n = (n + 1023) / 1024 * 1024;
    auto it = free_list.find(n);
    if (it != free_list.end()) { char* p = it->second; free_list.erase(it); return p; }
    char* p = base + off;
    off += n;
    if (off > peak) peak = off;
    return p;
  }
  void release(void* p, size_t n) { n = (n + 1023) / 1024 * 1024; free_list.emplace(n, (char*)p); }
};

}  // namespace

struct b2e_unet {
  b2e_unet_config cfg;
  int64_t max_batch = 0;
  // fp32-accurate mode (cfg.precision == 1): PL = 3, every activation is a split-f16 tensor with channel planes
  // [hi | lo | hi] (value = hi + lo) and every GEMM weight segment is packed [W_hi | W_hi | W_lo], so the unchanged
  // tcgen05 main loop computes x_hi W_hi + x_lo W_hi + x_hi W_lo with fp32 accumulation (~2^-17 relative error)
  int PL = 1;
  int temb_dim = 0, sumC = 0, heads_dim = 0;
  std::vector<void*> owned;
  struct PRec { std::string name; int64_t numel; int64_t fan_in; std::function<int(const float*, cudaStream_t)> set; };
  std::vector<PRec> params;
  std::unordered_map<std::string, int> pindex;
  ConvL conv_in, conv_out;
  bool in_im2col = false;
  // VQ decoder mode (b2e_vqdec_create): no time embedding, input = latent -> nearest-code quantisation + 1x1
  // post_quant_conv (one CUDA-core kernel) -> conv_in; output at sample_size << (n_blocks - 1)
  bool decoder = false;
  // VQ / KL encoder mode (b2e_vqenc_create): image -> conv_in -> down blocks -> mid block -> GroupNorm -> SiLU -> conv_out
  // (enc_q channels: latent, or 2 x latent moments) -> 1x1 quant_conv in fp32; output at sample_size >> (n_blocks - 1).
  // Split mode (encoder precision 1, PL = 3): the fp32-accurate forward of the decoder's split mode; quant_conv stays fp32
  bool encoder = false;
  // CLIP text encoder mode (b2e_clip_create): transformers CLIPTextModel - token + position embedding, pre-LN
  // transformer layers (causal 12-head self-attention on the fused kernel, quick-GELU MLP), final LayerNorm.  Split mode
  // (ccfg.precision == 1, PL = 3): the fp32-accurate forward, causal attention on the tiled fp32 kernel.
  // prep_text / encode_text, src/diffusion_utils.py:34-52
  bool clip = false;
  b2e_clip_config ccfg{};
  struct ClipL { LNL ln1, ln2; ConvL qkv, out, fc1, fc2; };
  std::vector<ClipL> clayers;
  LNL clip_final_ln;
  float *tok_emb = nullptr, *pos_emb = nullptr;
  const int64_t* in_ids = nullptr;
  // classifier mode (b2e_resnet_create): torchvision ResNet (BatchNorm folded into the convolutions by the host) ->
  // logits; backward: d(logits) -> d(image).  The loss network of ClassifierAttrFunc, src/attr_functions.py:222-257
  bool resnet = false;
  b2e_resnet_config rcfg{};
  struct RBlock { int nconv = 0; ConvL c[3]; int dg[3] = {-1, -1, -1}; int stride = 1; bool has_ds = false; int cin = 0, cout = 0; };
  std::vector<RBlock> rblocks;
  ConvL stem; int stem_dg = -1;
  float *fc_w = nullptr, *fc_b = nullptr;
  // face parser head (rcfg.head == 1): BiSeNet context path + feature fusion + output head (src/Segmentation/model.py)
  struct BiSe {
    ConvL arm32, arm16, head32, head16, ffm_blk, out_conv, out_cls;
    float *avg_w = nullptr, *avg_b = nullptr, *a32_w = nullptr, *a32_b = nullptr, *a16_w = nullptr, *a16_b = nullptr;
    float *f1_w = nullptr, *f2_w = nullptr;
  } bs;
  const float* in_dlogits = nullptr;
  int64_t* out_labels = nullptr;   // per call of b2e_resnet_forward_labels: argmax labels instead of logits
  // LPIPS mode (b2e_lpips_create): scaling layer -> VGG-16 features[0:30] (conv1_1 as a 1x1 convolution over the im2col
  // input, ReLU in every epilogue) -> distance head at relu1_2 .. relu5_3 against the reference's cached normalised
  // features; backward: d(dist) -> d(input).  The regulariser of the masked-prediction guidance (use_lpips)
  bool lpips = false;
  b2e_lpips_config lcfg{};
  std::vector<ConvL> vgg;                 // the thirteen convolutions; vgg[0] reads the im2col tensor
  float* lin_w[5] = {};                   // lin{k}.model.1.weight, C_k floats
  float* lp_const = nullptr;              // shift[3], scale[3], diag(1 / scale) (3 x 3): scaling layer and its adjoint
  size_t lp_ref_off[5] = {};             // reference cache (workspace offset 0): normalised tap features, fp32 [max_batch][HW_k][C_k]
  int64_t lp_ref_B = -1;                  // images in the cache (-1: none)
  bool lp_ref_mode = false;               // the forward fills the cache instead of computing distances
  const float* lp_mask = nullptr; int lp_mask_batched = 0;   // per call: input 1 - mask * x
  int enc_q = 0;
  float *qc_w = nullptr, *qc_b = nullptr;   // [enc_q][enc_q], [enc_q]
  float *codebook = nullptr, *pq_w = nullptr, *pq_b = nullptr;   // [n_codes][latent], [latent][latent], [latent]
  int n_codes = 0;
  // decoder gradient w.r.t. the latent (b2e_vqdec_backward): dgrad twins of every convolution, and a second op
  // list that walks the graph backwards over the activations the last forward left in the workspace
  std::vector<ConvL> dgrads;
  int conv_in_dg = -1, conv_out_dg = -1;
  bool grad = false;
  const float* in_dy = nullptr; float* out_dz = nullptr;   // per-call
  int64_t fwd_B = -1;                                      // batch of the forward whose activations are live
  NormL norm_out;
  float *te_w1 = nullptr, *te_b1 = nullptr, *te_w2 = nullptr, *te_b2 = nullptr, *tp_w = nullptr, *tp_b = nullptr;
  std::vector<ResnetL> resnets;
  std::vector<AttnL> attns;
  std::vector<XfL> xfs;
  const float* in_ctx = nullptr; int ctx_len = 0;   // per call: text conditioning (B, ctx_len, cross_attention_dim) fp32
  std::vector<ConvL> downs, ups;
  std::vector<Node> nodes;
  // program
  void* ws = nullptr; size_t ws_bytes = 0;
  int64_t cur_B = -1;
  struct Op { std::function<int(cudaStream_t)> fn; int kind; double flops; double bytes; std::string desc; };  // kind: 0 conv, 1 groupnorm, 2 attention, 3 other
  std::vector<Op> ops, bops;
  const float* in_x = nullptr; const int64_t* in_t = nullptr; float* out_eps = nullptr;  // per-call
  double flops = 0;
  size_t ws_need = 0;
  int build_error = 0;

  ~b2e_unet() { for (void* p : owned) cudaFree(p); }

  template <typename T> T* dmalloc(size_t n) {
    void* p = nullptr;
    if (cudaMalloc(&p, n * sizeof(T)) != cudaSuccess) { build_error = B2E_CUDA_ERROR; set_error("cudaMalloc(%zu) failed", n * sizeof(T)); return nullptr; }
    cudaMemset(p, 0, n * sizeof(T));
    owned.push_back(p);
    return (T*)p;
  }
  // fan_in: inputs per output unit (PyTorch default init bound 1/sqrt(fan_in)); 0 for norm layers
  void add_param(const std::string& name, int64_t numel, int64_t fan_in,
                 std::function<int(const float*, cudaStream_t)> fn) {
    pindex[name] = (int)params.size();
    params.push_back({name, numel, fan_in, std::move(fn)});
  }
  void add_f32(const std::string& name, float* dst, int64_t numel, int64_t fan_in = 0) {
    add_param(name, numel, fan_in, [dst, numel](const float* src, cudaStream_t st) -> int {
      B2E_CUDA(cudaMemcpyAsync(dst, src, numel * sizeof(float), cudaMemcpyDeviceToDevice, st));
      return (int)B2E_OK;
    });
  }
  // one K segment of a weight row: `plane_w` columns per plane starting at col_off; taps are tap_w * PL columns apart
  // fp32-accurate mode: every weight is packed times 2^10 and every convolution epilogue multiplies the accumulator by
  // 2^-10 (ConvEpilogue::acc_scale).  Exact, and it lifts the lo halves of the split weights (|w| 2^-11 ~ 1e-5 for a
  // typical |w| ~ 0.03) out of the fp16 subnormal range, where they would keep ~8 instead of 11 bits: the split weights
  // then carry ~22 bits like the split activations.  |w| * 2^10 <= 65504 holds for any |w| < 64.
  static constexpr float kSplitWScale = 1024.f;
  static int pack_w(int PL, const float* src, f16* w, int cout, int cin, int k, int tap_w, int row_len, int col_off,
                    int plane_w, cudaStream_t st, int ci0 = 0, int cin_total = 0) {
    if (PL == 1) return conv_pack_weight(src, w, cout, cin, k, tap_w, row_len, col_off, st, ci0, cin_total);
    int rc = conv_pack_weight(src, w, cout, cin, k, tap_w * 3, row_len, col_off, st, ci0, cin_total, 0, kSplitWScale);
    if (!rc) rc = conv_pack_weight(src, w, cout, cin, k, tap_w * 3, row_len, col_off + plane_w, st, ci0, cin_total, 0, kSplitWScale);
    if (!rc) rc = conv_pack_weight(src, w, cout, cin, k, tap_w * 3, row_len, col_off + 2 * plane_w, st, ci0, cin_total, 1, kSplitWScale);
    return rc;
  }
  // identity residual segment over the hi and lo planes (the repeated hi plane gets zero weights)
  static int fill_id(int PL, f16* w, int C, int row_len, int col_off, int plane_w) {
    int rc = conv_fill_identity(w, C, row_len, col_off, 0, PL == 3 ? kSplitWScale : 1.f);
    if (!rc && PL == 3) rc = conv_fill_identity(w, C, row_len, col_off + plane_w, 0, kSplitWScale);
    return rc;
  }
  // conv / linear weight that feeds the tcgen05 GEMM: packed f16 [cout_pad][k*k][cin_pad]
  // src0 > 0: the convolution reads TWO concatenated sources of src0 and cin - src0 channels (multiples of 64); in the
  // split mode every source carries its own [hi | lo | hi] planes, so the weight columns are packed per source
  ConvL make_conv(const std::string& name, int cin, int cout, int k, int cin_pad = 0, int res_c = 0, int src0 = 0, bool up2 = false) {
    ConvL c;
    c.cin = cin; c.cin_pad = cin_pad ? cin_pad : pad64(cin); c.cout = cout; c.k = k; c.cout_pad = conv_cout_pad(cout);
    c.res_c = res_c; c.row_len = PL * (k * k * c.cin_pad + res_c);
    c.w = dmalloc<f16>((size_t)c.cout_pad * c.row_len);
    c.b = dmalloc<float>(c.cout_pad);
    if (up2 && k == 3 && res_c == 0) {
      c.row_len_up2 = PL * 4 * c.cin_pad;
      c.w_up2 = dmalloc<f16>((size_t)4 * c.cout_pad * c.row_len_up2);
    }
    ConvL cc = c;
    ConvL dd;
    const int PL = this->PL;
    // (a <= 16-channel output, i.e. conv_out, receives its gradient as a 64-channel padded NHWC tensor)
    if (decoder || resnet || lpips) { c.dg = make_dgrad(cin, cout > 16 ? c.cout_pad : kConvBlockK, k); dd = dgrads[c.dg]; cc.dg = c.dg; }
    add_param(name + ".weight", (int64_t)cout * cin * k * k, (int64_t)cin * k * k, [cc, dd, PL, src0](const float* src, cudaStream_t st) {
      int rc;
      if (PL == 3 && src0 > 0 && cc.k == 1) {
        rc = pack_w(PL, src, cc.w, cc.cout, src0, 1, src0, cc.row_len, 0, src0, st, 0, cc.cin);
        if (!rc) rc = pack_w(PL, src, cc.w, cc.cout, cc.cin - src0, 1, cc.cin - src0, cc.row_len, 3 * src0, cc.cin - src0, st, src0, cc.cin);
      } else {
        rc = pack_w(PL, src, cc.w, cc.cout, cc.cin, cc.k, cc.cin_pad, cc.row_len, 0, cc.cin_pad, st);
      }
      if (!rc && cc.dg >= 0) rc = conv_pack_weight_dgrad(src, dd.w, cc.cout, cc.cin, cc.k, dd.cin_pad, dd.row_len, 0, st);
      for (int ph = 0; ph < 4 && !rc && cc.w_up2; ++ph) {
        f16* wp = cc.w_up2 + (size_t)ph * cc.cout_pad * cc.row_len_up2;
        if (PL == 1) {
          rc = conv_pack_weight_up2(src, wp, cc.cout, cc.cin, cc.cin_pad, cc.row_len_up2, 0, ph, st);
        } else {   // split mode: [W_hi | W_hi | W_lo] per tap, x 2^10 (as pack_w)
          rc = conv_pack_weight_up2(src, wp, cc.cout, cc.cin, 3 * cc.cin_pad, cc.row_len_up2, 0, ph, st, 0, kSplitWScale);
          if (!rc) rc = conv_pack_weight_up2(src, wp, cc.cout, cc.cin, 3 * cc.cin_pad, cc.row_len_up2, cc.cin_pad, ph, st, 0, kSplitWScale);
          if (!rc) rc = conv_pack_weight_up2(src, wp, cc.cout, cc.cin, 3 * cc.cin_pad, cc.row_len_up2, 2 * cc.cin_pad, ph, st, 1, kSplitWScale);
        }
      }
      return rc;
    });
    add_f32(name + ".bias", c.b, cout, (int64_t)cin * k * k);
    return c;
  }
  // dgrad twin of a stride-1 convolution with `cin` input channels whose output tensor has pitch `dy_pitch`:
  // a convolution dy (dy_pitch channels) -> dx (cin channels), zero bias; the weights are packed by the caller
  int make_dgrad(int cin, int dy_pitch, int k, int extra_k = 0) {
    ConvL d;
    d.cin = dy_pitch; d.cin_pad = dy_pitch; d.cout = cin; d.cout_pad = conv_cout_pad(cin); d.k = k;
    d.res_c = extra_k; d.row_len = k * k * dy_pitch + extra_k;
    d.w = dmalloc<f16>((size_t)d.cout_pad * d.row_len);
    d.b = dmalloc<float>(d.cout_pad);
    dgrads.push_back(d);
    return (int)dgrads.size() - 1;
  }
  NormL make_norm(const std::string& name, int C) {
    NormL n; n.C = C; n.g = dmalloc<float>(C); n.b = dmalloc<float>(C);
    add_f32(name + ".weight", n.g, C);
    add_f32(name + ".bias", n.b, C);
    return n;
  }
  int make_resnet(const std::string& name, int cin0, int cin1, int cout, bool with_temb = true) {
    ResnetL r;
    r.name = name; r.cin0 = cin0; r.cin1 = cin1; r.cout = cout;
    const int cin = cin0 + cin1;
    r.n1 = make_norm(name + ".norm1", cin);
    r.c1 = make_conv(name + ".conv1", cin, cout, 3);   // reads the compact GroupNorm output (pitch pad64(cin))
    if (with_temb) { r.temb_off = sumC; sumC += r.c1.cout_pad; }   // padded columns stay zero
    else r.temb_off = -1;
    r.n2 = make_norm(name + ".norm2", cout);
    // conv2 carries the block input as a fused 1x1 residual segment: conv_shortcut weights when the
    // channel count changes, the identity otherwise.  The segment reads the un-normalised block input(s)
    // at their own pitches: [pad64(cin0)][pad64(cin1)] columns.
    const int p0 = pad64(cin0), p1 = cin1 ? pad64(cin1) : 0;
    r.c2 = make_conv(name + ".conv2", cout, cout, 3, 0, p0 + p1);
    r.has_sc = cin != cout;
    if (r.has_sc) {
      r.c2.b2 = dmalloc<float>(r.c2.cout_pad);
      ConvL cc = r.c2;
      ConvL sd;
      if (decoder) { r.sc_dg = make_dgrad(cin, r.c2.cout_pad, 1); sd = dgrads[r.sc_dg]; }
      const int sc_dg = r.sc_dg;
      const int PL = this->PL;
      add_param(name + ".conv_shortcut.weight", (int64_t)cout * cin, cin, [cc, sd, sc_dg, cin, cin0, cin1, p0, p1, PL](const float* src, cudaStream_t st) {
        int rc = pack_w(PL, src, cc.w, cc.cout, cin0, 1, cin0, cc.row_len, PL * 9 * cc.cin_pad, p0, st, 0, cin);
        if (!rc && cin1) rc = pack_w(PL, src, cc.w, cc.cout, cin1, 1, cin1, cc.row_len, PL * (9 * cc.cin_pad + p0), p1, st, cin0, cin);
        if (!rc && sc_dg >= 0) rc = conv_pack_weight_dgrad(src, sd.w, cc.cout, cin, 1, sd.cin_pad, sd.row_len, 0, st);
        return rc;
      });
      add_f32(name + ".conv_shortcut.bias", r.c2.b2, cout, cin);
    } else if (r.c2.w) {
      if (cin1 && PL == 3) {   // identity over two split sources: rows [0, cin0) -> source 0, rows [cin0, cout) -> source 1
        if (fill_id(PL, r.c2.w, cin0, r.c2.row_len, PL * 9 * r.c2.cin_pad, p0) ||
            fill_id(PL, r.c2.w + (size_t)cin0 * r.c2.row_len, cin1, r.c2.row_len, PL * (9 * r.c2.cin_pad + p0), p1))
          build_error = B2E_CUDA_ERROR;
      } else if (fill_id(PL, r.c2.w, cout, r.c2.row_len, PL * 9 * r.c2.cin_pad, p0)) build_error = B2E_CUDA_ERROR;
    }
    resnets.push_back(r);
    return (int)resnets.size() - 1;
  }
  LNL make_ln(const std::string& name, int C) {
    LNL n; n.C = C; n.g = dmalloc<float>(C); n.b = dmalloc<float>(C);
    add_f32(name + ".weight", n.g, C);
    add_f32(name + ".bias", n.b, C);
    return n;
  }
  // token-wise linear layer = 1x1 convolution over NHWC pixels; res_c > 0 appends an identity residual segment
  ConvL make_linear(const std::string& name, int cin, int cout, bool bias, int res_c = 0) {
    ConvL c;
    c.cin = cin; c.cin_pad = pad64(cin); c.cout = cout; c.k = 1; c.cout_pad = conv_cout_pad(cout);
    c.res_c = res_c; c.row_len = PL * (c.cin_pad + res_c);
    c.w = dmalloc<f16>((size_t)c.cout_pad * c.row_len);
    c.b = dmalloc<float>(c.cout_pad);
    ConvL cc = c;
    const int PL = this->PL;
    add_param(name + ".weight", (int64_t)cout * cin, cin, [cc, PL](const float* src, cudaStream_t st) {
      return pack_w(PL, src, cc.w, cc.cout, cc.cin, 1, cc.cin_pad, cc.row_len, 0, cc.cin_pad, st);
    });
    if (bias) add_f32(name + ".bias", c.b, cout, cin);
    if (res_c && c.w && fill_id(PL, c.w, cout, c.row_len, PL * c.cin_pad, res_c)) build_error = B2E_CUDA_ERROR;
    return c;
  }
  // several bias-free projections of the same input fused into one GEMM: rows [i*cout, (i+1)*cout) = names[i]
  ConvL make_fused_linear(const std::string& base, const std::vector<std::string>& names, int cin, int cout, bool bias = false) {
    ConvL c;
    const int n = (int)names.size();
    c.cin = cin; c.cin_pad = pad64(cin); c.cout = n * cout; c.k = 1; c.cout_pad = conv_cout_pad(n * cout);
    c.row_len = c.cin_pad * PL;
    c.w = dmalloc<f16>((size_t)c.cout_pad * c.row_len);
    c.b = dmalloc<float>(c.cout_pad);
    const int PL = this->PL;
    for (int i = 0; i < n; ++i) {
      f16* wdst = c.w + (size_t)i * cout * c.row_len;
      const int rl = c.row_len, cp = c.cin_pad;
      add_param(base + "." + names[i] + ".weight", (int64_t)cout * cin, cin, [wdst, cout, cin, rl, cp, PL](const float* src, cudaStream_t st) {
        return pack_w(PL, src, wdst, cout, cin, 1, cp, rl, 0, cp, st);
      });
      if (bias && c.b) add_f32(base + "." + names[i] + ".bias", c.b + (size_t)i * cout, cout, cin);
    }
    return c;
  }
  int make_xformer(const std::string& name, int C, int heads, int ctx_dim) {
    XfL x;
    x.name = name; x.C = C; x.heads = heads; x.d = C / heads;
    x.gn = make_norm(name + ".norm", C);
    x.proj_in = make_linear(name + ".proj_in", C, C, true);
    const std::string tb = name + ".transformer_blocks.0";
    x.ln1 = make_ln(tb + ".norm1", C);
    x.ln2 = make_ln(tb + ".norm2", C);
    x.ln3 = make_ln(tb + ".norm3", C);
    x.qkv1 = make_fused_linear(tb + ".attn1", {"to_q", "to_k", "to_v"}, C, C);
    x.out1 = make_linear(tb + ".attn1.to_out.0", C, C, true, C);
    x.q2 = make_linear(tb + ".attn2.to_q", C, C, false);
    x.kv2 = make_fused_linear(tb + ".attn2", {"to_k", "to_v"}, ctx_dim, C);
    x.out2 = make_linear(tb + ".attn2.to_out.0", C, C, true, C);
    x.ff1 = make_linear(tb + ".ff.net.0.proj", C, 8 * C, true);
    x.ff2 = make_linear(tb + ".ff.net.2", 4 * C, C, true, C);
    x.proj_out = make_linear(name + ".proj_out", C, C, true, C);
    xfs.push_back(x);
    return (int)xfs.size() - 1;
  }
  int make_attn(const std::string& name, int C) {
    AttnL a;
    a.name = name; a.C = C; a.P = pad64(C);
    const int P = a.P;
    a.gn = make_norm(name + ".group_norm", C);
    // q, k, v fused into one [3P][P] GEMM weight (each projection padded to P rows / columns)
    a.qkv.cin = C; a.qkv.cin_pad = P; a.qkv.cout = 3 * P; a.qkv.cout_pad = conv_cout_pad(3 * P); a.qkv.k = 1;
    a.qkv.w = dmalloc<f16>((size_t)a.qkv.cout_pad * P * PL);
    a.qkv.b = dmalloc<float>(a.qkv.cout_pad);
    const int PL = this->PL;
    const char* nm[3] = {"to_q", "to_k", "to_v"};
    ConvL qd;
    if (decoder) { a.qkv_dg = make_dgrad(C, 2 * P, 1, P); qd = dgrads[a.qkv_dg]; }   // K = (dQ ++ dK) ++ residual segment dV
    const int qkv_dg = a.qkv_dg;
    for (int i = 0; i < 3; ++i) {
      f16* wdst = a.qkv.w + (size_t)i * P * P * PL;
      float* bdst = a.qkv.b + (size_t)i * P;
      add_param(name + "." + nm[i] + ".weight", (int64_t)C * C, C, [wdst, qd, qkv_dg, i, C, P, PL](const float* src, cudaStream_t st) {
        int rc = pack_w(PL, src, wdst, C, C, 1, C, P * PL, 0, P, st);
        if (!rc && qkv_dg >= 0) rc = conv_pack_weight_dgrad(src, qd.w, C, C, 1, P, qd.row_len, i * P, st);
        return rc;
      });
      add_f32(name + "." + nm[i] + ".bias", bdst, C, C);
    }
    a.qkv.row_len = P * PL;
    a.proj = make_conv(name + ".to_out.0", C, C, 1, 0, P);   // + identity residual segment
    if (a.proj.w && fill_id(PL, a.proj.w, C, a.proj.row_len, PL * a.proj.cin_pad, P)) build_error = B2E_CUDA_ERROR;
    attns.push_back(a);
    return (int)attns.size() - 1;
  }
};

namespace {

// VQModel.decode graph (diffusers Decoder): conv_in -> mid (resnet, single-head attention, resnet) -> per level,
// top-down, layers_per_block + 1 resnets (+ nearest x2 upsample + 3x3 conv) -> GroupNorm -> SiLU -> conv_out.
// cfg.block_out_channels is bottom-up as in the diffusers config ((128, 256, 512) for ldm-celebahq-256).
int build_model_decoder(b2e_unet* m) {
  const b2e_unet_config& c = m->cfg;
  const int nb = c.n_blocks, L = c.in_channels;
  const int top = c.block_out_channels[nb - 1];
  m->codebook = m->dmalloc<float>((size_t)(m->n_codes > 0 ? m->n_codes : 1) * L);
  m->pq_w = m->dmalloc<float>((size_t)L * L);
  m->pq_b = m->dmalloc<float>(L);
  if (m->n_codes > 0)   // num_vq_embeddings == 0: AutoencoderKL decode path (no quantiser)
    m->add_f32("quantize.embedding.weight", m->codebook, (int64_t)m->n_codes * L, -m->n_codes);   // U(-1/n, 1/n)
  m->add_f32("post_quant_conv.weight", m->pq_w, (int64_t)L * L, L);
  m->add_f32("post_quant_conv.bias", m->pq_b, L, L);
  m->in_im2col = true;
  {
    ConvL ci;
    const int PL = m->PL;
    ci.cin = ci.cin_pad = kConvBlockK; ci.cout = top; ci.k = 1; ci.cout_pad = conv_cout_pad(top); ci.row_len = kConvBlockK * PL;
    ci.w = m->dmalloc<f16>((size_t)ci.cout_pad * ci.row_len);
    ci.b = m->dmalloc<float>(ci.cout_pad);
    // dgrad twin: gradient w.r.t. the 64 im2col columns (9 * L real) = 1x1 convolution with the transposed weights
    m->conv_in_dg = m->make_dgrad(kConvBlockK, ci.cout_pad, 1);
    const ConvL cd = m->dgrads[m->conv_in_dg];
    m->add_param("decoder.conv_in.weight", (int64_t)top * L * 9, (int64_t)L * 9, [ci, cd, L, PL](const float* src, cudaStream_t st) {
      const float ws = PL == 3 ? b2e_unet::kSplitWScale : 1.f;
      int rc = conv_pack_weight(src, ci.w, ci.cout, L, 3, L, ci.row_len, 0, st, 0, 0, 0, ws);
      if (!rc && PL == 3) rc = conv_pack_weight(src, ci.w, ci.cout, L, 3, L, ci.row_len, kConvBlockK, st, 0, 0, 0, ws);
      if (!rc && PL == 3) rc = conv_pack_weight(src, ci.w, ci.cout, L, 3, L, ci.row_len, 2 * kConvBlockK, st, 0, 0, 1, ws);
      if (!rc) rc = conv_pack_weight_im2col_T(src, cd.w, ci.cout, L, cd.row_len, st);
      return rc;
    });
    m->add_f32("decoder.conv_in.bias", ci.b, top, (int64_t)L * 9);
    m->conv_in = ci;
  }
  int ch = top;
  m->nodes.push_back({N_RESNET, m->make_resnet("decoder.mid_block.resnets.0", ch, 0, ch, false)});
  m->nodes.push_back({N_ATTN, m->make_attn("decoder.mid_block.attentions.0", ch)});
  m->nodes.push_back({N_RESNET, m->make_resnet("decoder.mid_block.resnets.1", ch, 0, ch, false)});
  for (int i = 0; i < nb; ++i) {
    const int cout = c.block_out_channels[nb - 1 - i];
    const std::string base = "decoder.up_blocks." + std::to_string(i);
    for (int j = 0; j < c.layers_per_block + 1; ++j) {
      m->nodes.push_back({N_RESNET, m->make_resnet(base + ".resnets." + std::to_string(j), ch, 0, cout, false)});
      ch = cout;
    }
    if (i != nb - 1) {
      m->ups.push_back(m->make_conv(base + ".upsamplers.0.conv", ch, ch, 3, 0, 0, 0, true));
      m->nodes.push_back({N_UP, (int)m->ups.size() - 1});
    }
  }
  m->norm_out = m->make_norm("decoder.conv_norm_out", ch);
  m->conv_out = m->make_conv("decoder.conv_out", ch, c.out_channels, 3);
  m->conv_out_dg = m->conv_out.dg;
  return m->build_error;
}

// VQModel.encode / AutoencoderKL.encode graph (diffusers Encoder): conv_in -> per level layers_per_block resnets
// (+ pad (0,1,0,1) + 3x3 stride-2 conv) -> mid (resnet, single-head attention, resnet) -> GroupNorm -> SiLU ->
// conv_out -> quant_conv (1x1).  LDM.encode / SD.encode, src/diffusion_classes.py:27-30, 55-60.
int build_model_encoder(b2e_unet* m) {
  const b2e_unet_config& c = m->cfg;
  const int nb = c.n_blocks, cin = c.in_channels, c0 = c.block_out_channels[0], Q = m->enc_q;
  m->in_im2col = true;
  {
    // conv_in as a 1x1 convolution over the im2col input; split mode (PL = 3): [W_hi | W_hi | W_lo] x 2^10 over the
    // [hi | lo | hi] planes of the im2col tensor, as the decoder's conv_in
    ConvL ci;
    const int PL = m->PL;
    ci.cin = ci.cin_pad = kConvBlockK; ci.cout = c0; ci.k = 1; ci.cout_pad = conv_cout_pad(c0); ci.row_len = kConvBlockK * PL;
    ci.w = m->dmalloc<f16>((size_t)ci.cout_pad * ci.row_len);
    ci.b = m->dmalloc<float>(ci.cout_pad);
    m->add_param("encoder.conv_in.weight", (int64_t)c0 * cin * 9, (int64_t)cin * 9, [ci, cin, PL](const float* src, cudaStream_t st) {
      const float ws = PL == 3 ? b2e_unet::kSplitWScale : 1.f;
      int rc = conv_pack_weight(src, ci.w, ci.cout, cin, 3, cin, ci.row_len, 0, st, 0, 0, 0, ws);
      if (!rc && PL == 3) rc = conv_pack_weight(src, ci.w, ci.cout, cin, 3, cin, ci.row_len, kConvBlockK, st, 0, 0, 0, ws);
      if (!rc && PL == 3) rc = conv_pack_weight(src, ci.w, ci.cout, cin, 3, cin, ci.row_len, 2 * kConvBlockK, st, 0, 0, 1, ws);
      return rc;
    });
    m->add_f32("encoder.conv_in.bias", ci.b, c0, (int64_t)cin * 9);
    m->conv_in = ci;
  }
  int ch = c0;
  for (int i = 0; i < nb; ++i) {
    const int cout = c.block_out_channels[i];
    const std::string base = "encoder.down_blocks." + std::to_string(i);
    for (int j = 0; j < c.layers_per_block; ++j) {
      m->nodes.push_back({N_RESNET, m->make_resnet(base + ".resnets." + std::to_string(j), ch, 0, cout, false)});
      ch = cout;
    }
    if (i != nb - 1) {
      m->downs.push_back(m->make_conv(base + ".downsamplers.0.conv", ch, ch, 3));
      m->nodes.push_back({N_DOWN, (int)m->downs.size() - 1});
    }
  }
  m->nodes.push_back({N_RESNET, m->make_resnet("encoder.mid_block.resnets.0", ch, 0, ch, false)});
  m->nodes.push_back({N_ATTN, m->make_attn("encoder.mid_block.attentions.0", ch)});
  m->nodes.push_back({N_RESNET, m->make_resnet("encoder.mid_block.resnets.1", ch, 0, ch, false)});
  m->norm_out = m->make_norm("encoder.conv_norm_out", ch);
  m->conv_out = m->make_conv("encoder.conv_out", ch, Q, 3);
  m->qc_w = m->dmalloc<float>((size_t)Q * Q);
  m->qc_b = m->dmalloc<float>(Q);
  m->add_f32("quant_conv.weight", m->qc_w, (int64_t)Q * Q, Q);
  m->add_f32("quant_conv.bias", m->qc_b, Q, Q);
  return m->build_error;
}

// torchvision ResNet graph.  Parameter names are torchvision's convolution names with the eval-mode BatchNorm already
// folded in by the host ("layer1.0.conv1.weight" / ".bias", "layer1.0.downsample.0.weight" / ".bias", "conv1.*", "fc.*").
// Every block's last convolution carries the shortcut as a fused 1x1 residual K segment (identity or the downsample
// convolution on the - for stride 2, subsampled - block input); ReLU runs in the convolution epilogue.
int build_model_resnet(b2e_unet* m) {
  const b2e_resnet_config& c = m->rcfg;
  const int Cin = c.in_channels, W0 = c.width;
  const std::string pre = c.head == 1 ? "cp.resnet." : "";   // BiSeNet keeps its backbone under cp.resnet
  {
    // stem 7x7 stride 2 as a 1x1 convolution over a stride-2 im2col tensor (49 * Cin columns padded to a K-chunk multiple)
    // fp32-accurate forward (rcfg.precision == 1, PL = 3): forward activations are split tensors [hi | lo | hi] and the
    // forward weights are packed [W_hi | W_hi | W_lo] (x 2^10, undone in the epilogue) exactly as in the UNet's split mode,
    // so ReLU / max-pool masks agree with the fp32 reference; the backward pass (dgrad twins, gradients) stays on plain
    // f16 operands and reads its masks from the split activations.
    const int PL = m->PL;
    ConvL s;
    const int KP = pad64(49 * Cin);
    s.cin = s.cin_pad = KP; s.cout = W0; s.k = 1; s.cout_pad = conv_cout_pad(W0); s.row_len = KP * PL;
    s.w = m->dmalloc<f16>((size_t)s.cout_pad * KP * PL);
    s.b = m->dmalloc<float>(s.cout_pad);
    m->stem_dg = m->make_dgrad(KP, s.cout_pad, 1);   // gradient w.r.t. the im2col columns
    const ConvL sd = m->dgrads[m->stem_dg];
    m->add_param(pre + "conv1.weight", (int64_t)W0 * Cin * 49, (int64_t)Cin * 49, [s, sd, Cin, PL, KP](const float* src, cudaStream_t st) {
      const float ws = PL == 3 ? b2e_unet::kSplitWScale : 1.f;
      int rc = conv_pack_weight(src, s.w, s.cout, Cin, 7, Cin, s.row_len, 0, st, 0, 0, 0, ws);
      if (!rc && PL == 3) rc = conv_pack_weight(src, s.w, s.cout, Cin, 7, Cin, s.row_len, KP, st, 0, 0, 0, ws);
      if (!rc && PL == 3) rc = conv_pack_weight(src, s.w, s.cout, Cin, 7, Cin, s.row_len, 2 * KP, st, 0, 0, 1, ws);
      if (!rc) rc = conv_pack_weight_im2col_T(src, sd.w, s.cout, Cin, sd.row_len, st, 49);
      return rc;
    });
    m->add_f32(pre + "conv1.bias", s.b, W0, (int64_t)Cin * 49);
    m->stem = s;
  }
  const int expansion = c.bottleneck ? 4 : 1;
  int inpl = W0;
  for (int li = 0; li < 4; ++li) {
    const int planes = W0 << li;
    for (int bi = 0; bi < c.layers[li]; ++bi) {
      b2e_unet::RBlock rb;
      rb.stride = (bi == 0 && li > 0) ? 2 : 1;
      rb.cin = inpl; rb.cout = planes * expansion;
      rb.has_ds = rb.stride != 1 || inpl != rb.cout;
      const std::string base = pre + "layer" + std::to_string(li + 1) + "." + std::to_string(bi);
      // convolution list: bottleneck = 1x1, 3x3 (stride), 1x1 ; basic = 3x3 (stride), 3x3
      struct CS { int cin, cout, k; };
      std::vector<CS> cs;
      if (c.bottleneck) cs = {{inpl, planes, 1}, {planes, planes, 3}, {planes, rb.cout, 1}};
      else cs = {{inpl, planes, 3}, {planes, rb.cout, 3}};
      rb.nconv = (int)cs.size();
      for (int j = 0; j < rb.nconv; ++j) {
        const bool last = j == rb.nconv - 1;
        const std::string nm = base + ".conv" + std::to_string(j + 1);
        ConvL L;
        L.cin = cs[j].cin; L.cin_pad = pad64(cs[j].cin); L.cout = cs[j].cout; L.cout_pad = conv_cout_pad(cs[j].cout); L.k = cs[j].k;
        L.res_c = last ? pad64(inpl) : 0;
        L.row_len = m->PL * (L.k * L.k * L.cin_pad + L.res_c);
        L.w = m->dmalloc<f16>((size_t)L.cout_pad * L.row_len);
        L.b = m->dmalloc<float>(L.cout_pad);
        // dgrad twin; the FIRST convolution's twin also carries the shortcut gradient as a residual K segment
        // (identity, or the transposed downsample weights) so that d(block input) is ONE GEMM
        const int extra = j == 0 ? pad64(rb.cout) : 0;
        rb.dg[j] = m->make_dgrad(cs[j].cin, L.cout_pad, L.k, extra);
        const ConvL D = m->dgrads[rb.dg[j]];
        const int PLc = m->PL;
        m->add_param(nm + ".weight", (int64_t)L.cout * L.cin * L.k * L.k, (int64_t)L.cin * L.k * L.k, [L, D, PLc](const float* src, cudaStream_t st) {
          int rc = b2e_unet::pack_w(PLc, src, L.w, L.cout, L.cin, L.k, L.cin_pad, L.row_len, 0, L.cin_pad, st);
          if (!rc) rc = conv_pack_weight_dgrad(src, D.w, L.cout, L.cin, L.k, D.cin_pad, D.row_len, 0, st);
          return rc;
        });
        m->add_f32(nm + ".bias", L.b, L.cout, (int64_t)L.cin * L.k * L.k);
        rb.c[j] = L;
      }
      {
        const ConvL L = rb.c[rb.nconv - 1];
        const ConvL D0 = m->dgrads[rb.dg[0]];
        const int PLc = m->PL;
        const int seg = PLc * L.k * L.k * L.cin_pad;            // forward: residual segment starts here (all planes of the taps first)
        const int dseg = D0.k * D0.k * D0.cin_pad;              // backward twin of conv1: shortcut-gradient segment
        if (rb.has_ds) {
          rb.c[rb.nconv - 1].b2 = m->dmalloc<float>(L.cout_pad);
          const int cin = inpl, cout = rb.cout;
          m->add_param(base + ".downsample.0.weight", (int64_t)cout * cin, cin, [L, D0, seg, dseg, cin, cout, PLc](const float* src, cudaStream_t st) {
            int rc = b2e_unet::pack_w(PLc, src, L.w, cout, cin, 1, cin, L.row_len, seg, pad64(cin), st);
            if (!rc) rc = conv_pack_weight_dgrad(src, D0.w, cout, cin, 1, pad64(cout), D0.row_len, dseg, st);
            return rc;
          });
          m->add_f32(base + ".downsample.0.bias", rb.c[rb.nconv - 1].b2, cout, cin);
        } else if (L.w && D0.w) {
          if (b2e_unet::fill_id(PLc, L.w, rb.cout, L.row_len, seg, pad64(inpl)) || conv_fill_identity(D0.w, rb.cout, D0.row_len, dseg, 0))
            m->build_error = B2E_CUDA_ERROR;
        }
      }
      m->rblocks.push_back(rb);
      inpl = rb.cout;
    }
  }
  if (c.head == 1) {
    // BiSeNet: ConvBNReLU blocks (BatchNorm folded by the host) on the conv kernel; the 1x1 convolutions that act on
    // globally pooled vectors (conv_avg, the attention branches) are small fp32 matrices
    auto& bs = m->bs;
    const int c16 = W0 * 4, c32 = W0 * 8, c8 = W0 * 2, mid = 128;
    bs.arm32 = m->make_conv("cp.arm32.conv", c32, mid, 3);
    bs.arm16 = m->make_conv("cp.arm16.conv", c16, mid, 3);
    bs.head32 = m->make_conv("cp.conv_head32", mid, mid, 3);
    bs.head16 = m->make_conv("cp.conv_head16", mid, mid, 3);
    bs.ffm_blk = m->make_conv("ffm.convblk", c8 + mid, 256, 1, 0, 0, c8);   // reads feat8 (c8) ++ context path (mid)
    bs.out_conv = m->make_conv("conv_out.conv", 256, 256, 3);
    bs.out_cls = m->make_conv("conv_out.conv_out", 256, c.num_classes, 1);
    auto fcp = [&](const std::string& name, int K, int C, bool bias, float** w, float** b) {
      *w = m->dmalloc<float>((size_t)K * C);
      m->add_f32(name + ".weight", *w, (int64_t)K * C, C);
      if (bias) { *b = m->dmalloc<float>(K); m->add_f32(name + ".bias", *b, K, C); }
    };
    float* none = nullptr;
    fcp("cp.conv_avg", mid, c32, true, &bs.avg_w, &bs.avg_b);
    fcp("cp.arm32.conv_atten", mid, mid, true, &bs.a32_w, &bs.a32_b);
    fcp("cp.arm16.conv_atten", mid, mid, true, &bs.a16_w, &bs.a16_b);
    fcp("ffm.conv1", 64, 256, false, &bs.f1_w, &none);
    fcp("ffm.conv2", 256, 64, false, &bs.f2_w, &none);
    return m->build_error;
  }
  m->fc_w = m->dmalloc<float>((size_t)c.num_classes * inpl);
  m->fc_b = m->dmalloc<float>(c.num_classes);
  m->add_f32("fc.weight", m->fc_w, (int64_t)c.num_classes * inpl, inpl);
  m->add_f32("fc.bias", m->fc_b, c.num_classes, inpl);
  return m->build_error;
}

// Launch list of the classifier for batch B: forward (activations kept: every ReLU output is needed by the backward pass)
// and backward (d logits -> d image).  Same arena / plan machinery as the UNet.
int build_program_resnet(b2e_unet* m, int B, void* ws, size_t ws_bytes, size_t* need) {
  const b2e_resnet_config& c = m->rcfg;
  Arena ar;
  ar.reset(ws, ws_bytes);
  const bool dry = ar.dry;
  std::vector<b2e_unet::Op> fwd, bwd;
  std::vector<b2e_unet::Op>* cur = &fwd;
  double flops = 0;
  int rc = B2E_OK;
  const int PL = m->PL;     // planes of the FORWARD activations (3: split tensors of the fp32-accurate forward); gradients: 1
  auto talloc = [&](int N, int H, int W, int C, int planes = 1) {
    Tensor t; t.N = N; t.H = H; t.W = W; t.C = C; t.Cr = C; t.bytes = (size_t)N * H * W * C * planes * sizeof(f16);
    t.p = (f16*)ar.alloc(t.bytes);
    return t;
  };
  const size_t split_bytes = (size_t)kNumSMs * kConvBlockM * 128 * sizeof(float);
  float* split_ws = (float*)ar.alloc(split_bytes);
  int* split_cnt = (int*)ar.alloc(sizeof(int) * 1024);
  if (!dry) cudaMemset(split_cnt, 0, sizeof(int) * 1024);
  // y = [relu](conv_{k, stride}(x) [+ W_r r0] + bias [+ bias2]); stride 2: symmetric padding 1 (torchvision)
  auto conv = [&](const ConvL& L, const Tensor& x, int stride, bool relu, const Tensor* r0, Tensor* out, const char* what,
                  const Tensor* x1 = nullptr) {
    if (rc) return;
    const int Ho = x.H / stride, Wo = x.W / stride;
    const int xc = x.C + (x1 ? x1->C : 0);
    *out = talloc(B, Ho, Wo, L.cout_pad, PL);
    const double fl = 2.0 * B * Ho * Wo * (double)L.cout_pad * (L.k * L.k * xc + L.res_c) * PL;
    flops += fl;
    if (dry) return;
    if (PL * (L.k * L.k * xc + L.res_c) != L.row_len || L.res_c != (r0 ? r0->C : 0)) {
      rc = B2E_INVALID_ARG; set_error("resnet: operand widths do not match the packed weights (%s)", what); return;
    }
    ConvDesc d;
    d.s0 = ConvSrc{x.p, x.C * PL};
    if (x1) d.s1 = ConvSrc{x1->p, x1->C * PL};
    if (r0) d.r0 = ConvSrc{r0->p, r0->C * PL};
    d.out_planes = PL;
    d.N = B; d.H = x.H; d.W = x.W; d.ksize = L.k; d.stride = stride; d.stride2_pad1 = 1;
    d.w_packed = L.w; d.Cout = L.cout_pad; d.out_f16 = out->p;
    d.split_ws = split_ws; d.split_ws_bytes = split_bytes; d.split_counters = split_cnt;
    ConvPlan pl;
    rc = conv_plan_build(&pl, d);
    if (rc) return;
    ConvEpilogue ep;
    ep.bias = L.b; ep.bias2 = L.b2; ep.relu = relu ? 1 : 0;
    if (PL == 3) ep.acc_scale = 1.f / b2e_unet::kSplitWScale;
    char desc[160];
    snprintf(desc, sizeof(desc), "%s: conv%dx%d s%d %dx%d cin%d res%d cout%d bn%d%s%s", what, L.k, L.k, stride, x.H, x.W, x.C, L.res_c,
             L.cout, pl.block_n, pl.halo ? " halo" : pl.pair ? " pair" : "", relu ? " +relu" : "");
    cur->push_back({[pl, ep](cudaStream_t st) { return conv_launch(pl, ep, st); }, 0, pl.flops, 0.0, desc});
  };
  auto ew = [&](std::function<int(cudaStream_t)> fn, double bytes, const char* what) {
    if (!dry && !rc) cur->push_back({std::move(fn), 3, 0.0, bytes, what});
  };
  // the stride of a block sits on the 3x3 convolution of a bottleneck (torchvision v1.5) / the first one of a basic block
  auto cstride = [](const b2e_unet::RBlock& rb, int j) { return (rb.nconv == 3 ? j == 1 : j == 0) ? rb.stride : 1; };

  // ---------------- forward
  const int S = c.input_size, Cin = c.in_channels, KP = m->stem.cin_pad;
  Tensor cols = talloc(B, S / 2, S / 2, KP, PL);
  ew([m, cols, B, Cin, S, KP, PL](cudaStream_t st) { return im2col7s2_launch(m->in_x, cols.p, B, Cin, S, S, KP, st, PL); },
     (double)B * S * S * Cin * 4.0 + (double)cols.bytes, "stem im2col (7x7 stride 2)");
  Tensor y1, y2;
  conv(m->stem, cols, 1, true, nullptr, &y1, "stem");
  y2 = talloc(B, y1.H / 2, y1.W / 2, y1.C, PL);
  uint8_t* pool_idx = (uint8_t*)ar.alloc((size_t)B * y2.H * y2.W * y2.C);
  ew([y1, y2, pool_idx, B, PL](cudaStream_t st) { return maxpool3s2_launch(y1.p, y2.p, pool_idx, B, y1.H, y1.W, y1.C, st, PL); },
     1.25 * (double)y1.bytes + (double)y2.bytes, "maxpool 3x3 stride 2");
  struct BSave { Tensor x, xs, a[3]; };
  std::vector<BSave> saves(m->rblocks.size());
  std::vector<Tensor> layer_out;
  Tensor h = y2;
  for (size_t bi = 0; bi < m->rblocks.size() && !rc; ++bi) {
    const b2e_unet::RBlock& rb = m->rblocks[bi];
    BSave& sv = saves[bi];
    sv.x = h;
    // shortcut operand at the block's output resolution
    sv.xs = h;
    if (rb.stride == 2) {
      sv.xs = talloc(B, h.H / 2, h.W / 2, h.C, PL);
      const Tensor hh = h, xs = sv.xs;
      ew([hh, xs, B, PL](cudaStream_t st) { return subsample2x_launch(hh.p, xs.p, B, xs.H, xs.W, xs.C * PL, st); }, 2.0 * (double)xs.bytes,
         "shortcut subsample");
    }
    Tensor t = h;
    for (int j = 0; j < rb.nconv; ++j) {
      const bool last = j == rb.nconv - 1;
      // the stride sits on the 3x3 convolution (torchvision v1.5 bottleneck) / on the first convolution of a basic block
      const int stride = cstride(rb, j);
      conv(rb.c[j], t, stride, true, last ? &sv.xs : nullptr, &sv.a[j], last ? "block out" : "block conv");
      t = sv.a[j];
    }
    h = t;
    layer_out.push_back(h);
  }
  const int HWl = h.H * h.W, Cl = h.C, K = c.num_classes;
  // face-parser head: what its backward pass needs from the forward
  struct HeadSave {
    Tensor feat8, feat16, feat32, f32, h32, f16, cp8, ff, o1, o2;
    float *p32 = nullptr, *avg = nullptr, *q32 = nullptr, *att32 = nullptr, *q16 = nullptr, *att16 = nullptr, *pf = nullptr, *t1 = nullptr,
          *attf = nullptr;
  } hs;
  if (!rc && c.head == 1) {
    // ---- BiSeNet: context path (attention refinement on feat16 / feat32 + global context), feature fusion with the
    // 1/8 backbone feature, output head, bilinear (align_corners) upsampling to the input resolution -> fp32 NCHW logits
    const auto& bs = m->bs;
    int nb = 0;
    Tensor feat8, feat16, feat32;
    for (int li = 0; li < 4; ++li) {
      nb += c.layers[li];
      if (li == 1) feat8 = layer_out[nb - 1];
      if (li == 2) feat16 = layer_out[nb - 1];
      if (li == 3) feat32 = layer_out[nb - 1];
    }
    auto fbuf = [&](int n) { return (float*)ar.alloc(sizeof(float) * B * n); };
    auto pool = [&](const Tensor& t, float* dst) {
      const Tensor tt = t;
      ew([tt, dst, B, PL](cudaStream_t st) { return avgpool_launch(tt.p, dst, B, tt.H * tt.W, tt.C, st, PL); }, (double)tt.bytes, "global average pool");
    };
    auto fc = [&](const float* x, const float* w, const float* b, float* out, int C, int Kk, int act, const char* what) {
      ew([x, w, b, out, B, C, Kk, act](cudaStream_t st) { return fc_act_launch(x, w, b, out, B, C, Kk, act, st); }, 4.0 * Kk * C, what);
    };
    auto affine = [&](const Tensor& x, const float* a, const float* b, const Tensor* y, Tensor* out, const char* what) {
      *out = talloc(B, x.H, x.W, x.C, PL);
      const Tensor xx = x, oo = *out;
      const f16* yp = y ? y->p : nullptr;
      ew([xx, a, b, yp, oo, B, PL](cudaStream_t st) { return chan_affine_launch(xx.p, a, b, yp, oo.p, B, xx.H * xx.W, xx.C, st, PL); },
         (y ? 3.0 : 2.0) * (double)xx.bytes, what);
    };
    auto up2 = [&](const Tensor& x, Tensor* out) {
      *out = talloc(B, x.H * 2, x.W * 2, x.C, PL);
      const Tensor xx = x, oo = *out;
      ew([xx, oo, B, PL](cudaStream_t st) { return upsample2x_launch(xx.p, oo.p, B, xx.H, xx.W, xx.C * PL, st); }, 1.25 * (double)oo.bytes, "nearest upsample x2");
    };
    const int mid = 128;
    hs.feat8 = feat8; hs.feat16 = feat16; hs.feat32 = feat32;
    hs.p32 = fbuf(feat32.C); hs.avg = fbuf(mid); hs.q32 = fbuf(mid); hs.att32 = fbuf(mid); hs.q16 = fbuf(mid); hs.att16 = fbuf(mid);
    hs.pf = fbuf(256); hs.t1 = fbuf(64); hs.attf = fbuf(256);
    Tensor sum32, up32, sum16, up16, fo;
    pool(feat32, hs.p32);
    fc(hs.p32, bs.avg_w, bs.avg_b, hs.avg, feat32.C, mid, 1, "conv_avg (1x1 on the pooled feature)");
    conv(bs.arm32, feat32, 1, true, nullptr, &hs.f32, "arm32.conv");
    pool(hs.f32, hs.q32);
    fc(hs.q32, bs.a32_w, bs.a32_b, hs.att32, mid, mid, 2, "arm32 attention");
    affine(hs.f32, hs.att32, hs.avg, nullptr, &sum32, "arm32: feat * attention + global context");
    up2(sum32, &up32);
    conv(bs.head32, up32, 1, true, nullptr, &hs.h32, "conv_head32");
    conv(bs.arm16, feat16, 1, true, nullptr, &hs.f16, "arm16.conv");
    pool(hs.f16, hs.q16);
    fc(hs.q16, bs.a16_w, bs.a16_b, hs.att16, mid, mid, 2, "arm16 attention");
    affine(hs.f16, hs.att16, nullptr, &hs.h32, &sum16, "arm16: feat * attention + feat32_up");
    up2(sum16, &up16);
    conv(bs.head16, up16, 1, true, nullptr, &hs.cp8, "conv_head16");
    conv(bs.ffm_blk, feat8, 1, true, nullptr, &hs.ff, "ffm.convblk (concat fused)", &hs.cp8);
    pool(hs.ff, hs.pf);
    fc(hs.pf, bs.f1_w, nullptr, hs.t1, 256, 64, 1, "ffm.conv1");
    fc(hs.t1, bs.f2_w, nullptr, hs.attf, 64, 256, 3, "ffm.conv2 (1 + sigmoid)");
    affine(hs.ff, hs.attf, nullptr, nullptr, &fo, "ffm: feat * (1 + attention)");
    conv(bs.out_conv, fo, 1, true, nullptr, &hs.o1, "conv_out.conv");
    conv(bs.out_cls, hs.o1, 1, false, nullptr, &hs.o2, "conv_out.conv_out");
    if (!rc) {
      const Tensor oo = hs.o2;
      // b2e_resnet_forward_labels sets out_labels for its call: the upsampled logits go straight into their argmax
      ew([m, oo, B, K, S, PL](cudaStream_t st) {
           return m->out_labels ? bilinear_ac_argmax_launch(oo.p, m->out_labels, B, oo.H, oo.W, oo.C, K, S, S, st, PL)
                                : bilinear_ac_launch(oo.p, m->out_eps, B, oo.H, oo.W, oo.C, K, S, S, st, PL); },
         (double)oo.bytes + 4.0 * B * K * S * S, "bilinear upsample (align_corners) -> logits");
    }
  }
  float* feat = (float*)ar.alloc(sizeof(float) * B * Cl);
  if (!rc && c.head == 0) {
    const Tensor hl = h;
    ew([m, hl, feat, B, HWl, Cl, K, PL](cudaStream_t st) { return avgpool_fc_launch(hl.p, feat, m->fc_w, m->fc_b, m->out_eps, B, HWl, Cl, K, st, PL); },
       (double)hl.bytes, "global average pool + fc");
  }
  // ---------------- backward: d(logits) -> d(image)
  if (!rc && m->grad) {
    cur = &bwd;
    Tensor g;   // gradient w.r.t. the PRE-activation of the current block output
    // gradients that reach a backbone feature from a second consumer (face parser: feat8 -> ffm, feat16 -> arm16):
    // key = index of the block whose INPUT is that feature; value = (tensor, channel offset of the window)
    std::map<int, std::pair<Tensor, int>> extra;
    auto dconv = [&](int dg, const Tensor& dy, const Tensor* r0, Tensor* dx, const char* what) {
      // dx = conv_{k, stride 1}(dy; flipped / transposed weights) [+ residual segment r0]
      if (rc) return;
      const ConvL& D = m->dgrads[dg];
      *dx = talloc(B, dy.H, dy.W, D.cout_pad);
      const double fl = 2.0 * B * dy.H * dy.W * (double)D.cout_pad * D.row_len;
      flops += fl;
      if (dry) return;
      if (D.k * D.k * dy.C + D.res_c != D.row_len || (r0 ? r0->C : 0) != D.res_c) {
        rc = B2E_INVALID_ARG; set_error("resnet backward: operand widths do not match (%s)", what); return;
      }
      ConvDesc d;
      d.s0 = ConvSrc{dy.p, dy.C};
      if (r0) d.r0 = ConvSrc{r0->p, r0->C};
      d.N = B; d.H = dy.H; d.W = dy.W; d.ksize = D.k; d.stride = 1;
      d.w_packed = D.w; d.Cout = D.cout_pad; d.out_f16 = dx->p;
      d.split_ws = split_ws; d.split_ws_bytes = split_bytes; d.split_counters = split_cnt;
      ConvPlan pl;
      rc = conv_plan_build(&pl, d);
      if (rc) return;
      char desc[160];
      snprintf(desc, sizeof(desc), "%s: dgrad conv%dx%d %dx%d cin%d res%d cout%d", what, D.k, D.k, dy.H, dy.W, dy.C, D.res_c, D.cout);
      cur->push_back({[pl](cudaStream_t st) { return conv_launch(pl, ConvEpilogue{}, st); }, 0, pl.flops, 0.0, desc});
    };
    auto relu_mask = [&](Tensor& gt, const Tensor& y) {   // in place: gt *= (y > 0); y = forward activation (PL planes)
      const Tensor gg = gt, yy = y;
      ew([gg, yy, PL](cudaStream_t st) { return relu_bwd_launch(gg.p, yy.p, gg.p, (int64_t)(gg.bytes / sizeof(f16)), st, PL, gg.C); },
         3.0 * (double)gt.bytes, "relu backward");
    };
    auto zero_up = [&](const Tensor& t) {
      Tensor u = talloc(B, t.H * 2, t.W * 2, t.C);
      const Tensor tt = t;
      ew([tt, u, B](cudaStream_t st) { return zero_upsample2x_launch(tt.p, u.p, B, tt.H, tt.W, tt.C, st); }, 1.25 * (double)u.bytes,
         "zero insertion (stride-2 gradient)");
      return u;
    };
    // gradient scale record (grad_scale_launch): keeps the f16 gradients in range; every backward op is linear in g
    float* gsc = (float*)ar.alloc(sizeof(float) * 4);
    if (!dry) cudaMemset(gsc, 0, sizeof(float) * 4);
    {
      // expected magnitude of the first f16 gradient tensor relative to max|d(logits)|: the pooling / fc adjoint of the
      // classifier (1 / HW, weights ~ 1 / sqrt(C)), the bilinear adjoint of the parser (sums (S / Hlow)^2 logit gradients)
      const float mult = c.head == 0 ? 1.f / ((float)HWl * sqrtf((float)Cl)) : (float)(S / (S / 8)) * (float)(S / (S / 8));
      const int64_t n = c.head == 0 ? (int64_t)B * K : (int64_t)B * K * S * S;
      ew([m, gsc, n, mult](cudaStream_t st) { return grad_scale_launch(m->in_dlogits, n, gsc, mult, st); }, 4.0 * (double)n,
         "max|d(logits)| -> power-of-two gradient scale");
    }
    if (c.head == 0) {
      float* dfeat = (float*)ar.alloc(sizeof(float) * B * Cl);
      g = talloc(B, h.H, h.W, h.C);
      const Tensor hl = h, gg = g;
      ew([m, hl, gg, dfeat, gsc, B, HWl, Cl, K, PL](cudaStream_t st) {
           return avgpool_fc_bwd_launch(m->in_dlogits, m->fc_w, dfeat, hl.p, gg.p, B, HWl, Cl, K, st, gsc, PL); },
         2.0 * (double)hl.bytes, "fc + average pool backward (+ relu mask)");
    } else {
      // ---- face parser head backward: d(logits) (B, K, S, S) -> gradients at feat8 / feat16 / feat32
      const auto& bs = m->bs;
      auto fbuf = [&](int n) { return (float*)ar.alloc(sizeof(float) * B * n); };
      auto dot = [&](const Tensor& x, const Tensor* y, float* out, float scale, const char* what) {
        const Tensor xx = x;
        const f16* yp = y ? y->p : nullptr;
        ew([xx, yp, out, B, scale, PL](cudaStream_t st) { return chan_dot_launch(xx.p, yp, out, B, xx.H * xx.W, xx.C, scale, st, PL); },
           (y ? 2.0 : 1.0) * (double)xx.bytes, what);
      };
      auto vact = [&](const float* gv, const float* a, float* out, int n, int mode) {
        ew([gv, a, out, n, mode](cudaStream_t st) { return vec_act_bwd_launch(gv, a, out, n, mode, st); }, 12.0 * n, "attention activation backward");
      };
      auto fct = [&](const float* gv, const float* w, float* out, int C, int Kk, float scale) {
        ew([gv, w, out, B, C, Kk, scale](cudaStream_t st) { return fc_t_launch(gv, w, out, B, C, Kk, scale, st); }, 4.0 * C * Kk, "transposed 1x1 on pooled vector");
      };
      auto affine = [&](const Tensor& x, const float* a, const float* b, Tensor* out, const char* what) {
        *out = talloc(B, x.H, x.W, x.C);
        const Tensor xx = x, oo = *out;
        ew([xx, a, b, oo, B](cudaStream_t st) { return chan_affine_launch(xx.p, a, b, nullptr, oo.p, B, xx.H * xx.W, xx.C, st); },
           2.0 * (double)xx.bytes, what);
      };
      auto merge = [&](const Tensor* gt, const Tensor* e, int e_off, const Tensor* y, Tensor* out, int C, int H, int W, const char* what) {
        *out = talloc(B, H, W, C);
        const Tensor oo = *out;
        const f16* gp = gt ? gt->p : nullptr; const f16* ep = e ? e->p : nullptr; const f16* yp = y ? y->p : nullptr;
        const int epitch = e ? e->C : 0;
        ew([gp, ep, epitch, e_off, yp, oo, B, PL](cudaStream_t st) {
             return grad_merge_launch(gp, ep, epitch, e_off, yp, oo.p, (int64_t)B * oo.H * oo.W, oo.C, st, PL); }, 3.0 * (double)oo.bytes, what);
      };
      auto down2 = [&](const Tensor& dy, Tensor* dx) {
        *dx = talloc(B, dy.H / 2, dy.W / 2, dy.C);
        const Tensor dd = dy, xx = *dx;
        ew([dd, xx, B](cudaStream_t st) { return downsum2x_launch(dd.p, xx.p, B, xx.H, xx.W, xx.C, st); }, 1.25 * (double)dd.bytes, "nearest upsample backward");
      };
      const int mid = 128;
      const float i8 = 1.f / (float)(hs.ff.H * hs.ff.W), i16 = 1.f / (float)(hs.f16.H * hs.f16.W), i32 = 1.f / (float)(hs.f32.H * hs.f32.W);
      Tensor g_o2 = talloc(B, hs.o2.H, hs.o2.W, hs.o2.C), g_o1, g_fo, g_ff, g_cat, g_cp8, g_up16, g_sum16, g_h32, g_f16, e16, g_up32,
             g_sum32, g_f32, e32, g32;
      {
        const Tensor oo = g_o2;
        ew([m, oo, gsc, B, K, S](cudaStream_t st) { return bilinear_ac_bwd_launch(m->in_dlogits, oo.p, B, oo.H, oo.W, oo.C, K, S, S, st, gsc); },
           4.0 * B * K * S * S, "bilinear upsample backward");
      }
      dconv(bs.out_cls.dg, g_o2, nullptr, &g_o1, "conv_out.conv_out");
      relu_mask(g_o1, hs.o1);
      dconv(bs.out_conv.dg, g_o1, nullptr, &g_fo, "conv_out.conv");
      // feature fusion: fo = ff * a, a = 1 + sigmoid(W2 relu(W1 mean(ff)))
      float *ga = fbuf(256), *gz2 = fbuf(256), *gt1 = fbuf(64), *gt1m = fbuf(64), *gpf = fbuf(256);
      dot(g_fo, &hs.ff, ga, 1.f, "ffm: d(attention)");
      vact(ga, hs.attf, gz2, B * 256, 2);
      fct(gz2, bs.f2_w, gt1, 64, 256, 1.f);
      vact(gt1, hs.t1, gt1m, B * 64, 0);
      fct(gt1m, bs.f1_w, gpf, 256, 64, i8);
      affine(g_fo, hs.attf, gpf, &g_ff, "ffm: d(feat) = g * (1 + attention) + pooled path");
      relu_mask(g_ff, hs.ff);
      dconv(bs.ffm_blk.dg, g_ff, nullptr, &g_cat, "ffm.convblk");     // channels [0, c8) -> feat8, [c8, c8 + 128) -> cp8
      const int c8 = hs.feat8.C;
      merge(nullptr, &g_cat, c8, &hs.cp8, &g_cp8, mid, hs.cp8.H, hs.cp8.W, "d(cp8) window + relu mask");
      dconv(bs.head16.dg, g_cp8, nullptr, &g_up16, "conv_head16");
      down2(g_up16, &g_sum16);
      // sum16 = f16 * att16 + h32
      merge(&g_sum16, nullptr, 0, &hs.h32, &g_h32, mid, hs.h32.H, hs.h32.W, "d(feat32_up) + relu mask");
      float *ga16 = fbuf(mid), *gz16 = fbuf(mid), *gq16 = fbuf(mid);
      dot(g_sum16, &hs.f16, ga16, 1.f, "arm16: d(attention)");
      vact(ga16, hs.att16, gz16, B * mid, 1);
      fct(gz16, bs.a16_w, gq16, mid, mid, i16);
      affine(g_sum16, hs.att16, gq16, &g_f16, "arm16: d(feat)");
      relu_mask(g_f16, hs.f16);
      dconv(bs.arm16.dg, g_f16, nullptr, &e16, "arm16.conv");
      // feat32_up = relu(conv_head32(up(sum32)))
      dconv(bs.head32.dg, g_h32, nullptr, &g_up32, "conv_head32");
      down2(g_up32, &g_sum32);
      // sum32 = f32 * att32 + avg ; avg = relu(W_avg mean(feat32) + b)
      float *gavg = fbuf(mid), *gavgm = fbuf(mid), *gp32 = fbuf(hs.feat32.C), *ga32 = fbuf(mid), *gz32 = fbuf(mid), *gq32 = fbuf(mid);
      dot(g_sum32, nullptr, gavg, 1.f, "d(global context)");
      vact(gavg, hs.avg, gavgm, B * mid, 0);
      fct(gavgm, bs.avg_w, gp32, hs.feat32.C, mid, i32);
      dot(g_sum32, &hs.f32, ga32, 1.f, "arm32: d(attention)");
      vact(ga32, hs.att32, gz32, B * mid, 1);
      fct(gz32, bs.a32_w, gq32, mid, mid, i32);
      affine(g_sum32, hs.att32, gq32, &g_f32, "arm32: d(feat)");
      relu_mask(g_f32, hs.f32);
      dconv(bs.arm32.dg, g_f32, nullptr, &e32, "arm32.conv");
      affine(e32, nullptr, gp32, &g32, "d(feat32) = arm32 path + pooled path");
      relu_mask(g32, hs.feat32);
      g = g32;
      extra[c.layers[0] + c.layers[1] + c.layers[2]] = {e16, 0};   // feat16 = input of layer4's first block
      extra[c.layers[0] + c.layers[1]] = {g_cat, 0};                // feat8  = input of layer3's first block
    }
    for (int bi = (int)m->rblocks.size() - 1; bi >= 0 && !rc; --bi) {
      const b2e_unet::RBlock& rb = m->rblocks[bi];
      const BSave& sv = saves[bi];
      // g = d/d(pre-activation of the block output).  Walk the convolutions backwards; the first convolution's twin
      // adds the shortcut gradient through its residual segment.
      Tensor gs = g;                     // shortcut gradient operand at the block INPUT resolution
      if (rb.stride == 2) gs = zero_up(g);
      Tensor d = g;
      for (int j = rb.nconv - 1; j >= 1; --j) {
        const int stride = cstride(rb, j);
        Tensor dy = d;
        if (stride == 2) dy = zero_up(d);
        Tensor dx;
        dconv(rb.dg[j], dy, nullptr, &dx, "block");
        relu_mask(dx, sv.a[j - 1]);
        d = dx;
      }
      {
        const int stride0 = cstride(rb, 0);
        Tensor dy = d;
        if (stride0 == 2) dy = zero_up(d);
        Tensor dx;
        dconv(rb.dg[0], dy, &gs, &dx, "block in");
        // the block input is the previous block's ReLU output (or the max-pool output, whose mask is applied there);
        // a backbone feature with a second consumer collects that gradient before the mask
        auto ex = extra.find(bi);
        if (ex != extra.end() && !rc) {
          const Tensor gd = dx, ee = ex->second.first, yy = sv.x;
          const int eoff = ex->second.second;
          Tensor merged = talloc(B, dx.H, dx.W, dx.C);
          ew([gd, ee, eoff, yy, merged, B, PL](cudaStream_t st) {
               return grad_merge_launch(gd.p, ee.p, ee.C, eoff, yy.p, merged.p, (int64_t)B * merged.H * merged.W, merged.C, st, PL); },
             4.0 * (double)merged.bytes, "gradient merge (second consumer) + relu mask");
          dx = merged;
        } else if (bi > 0) {
          relu_mask(dx, sv.x);
        }
        g = dx;
      }
    }
    if (!rc) {
      // max pool (+ the stem's ReLU mask) -> stem dgrad w.r.t. the im2col columns -> col2im -> fp32 NCHW image gradient
      Tensor gy1 = talloc(B, y1.H, y1.W, y1.C), dcols;
      const Tensor gg = g;
      ew([y1, pool_idx, gg, gy1, B, PL](cudaStream_t st) { return maxpool3s2_bwd_launch(y1.p, pool_idx, gg.p, gy1.p, B, y1.H, y1.W, y1.C, st, PL); },
         3.0 * (double)y1.bytes, "maxpool backward (+ stem relu mask)");
      dconv(m->stem_dg, gy1, nullptr, &dcols, "stem");
      if (!rc) {
        const Tensor dc = dcols;
        ew([m, dc, gsc, B, Cin, S, KP](cudaStream_t st) { return col2im7s2_launch(dc.p, m->out_dz, B, Cin, S, S, KP, st, gsc); },
           (double)dc.bytes + 4.0 * B * Cin * S * S, "stem col2im (image gradient)");
      }
    }
    cur = &fwd;
  }
  if (rc) return rc;
  if (need) *need = ar.peak;
  if (!dry) {
    B2E_REQUIRE(ar.peak <= ws_bytes, B2E_WORKSPACE_TOO_SMALL, "resnet: workspace too small (%zu > %zu)", ar.peak, ws_bytes);
    m->ops = std::move(fwd);
    m->bops = std::move(bwd);
    m->fwd_B = -1;
    m->cur_B = B;
  }
  m->flops = flops;
  return B2E_OK;
}

// LPIPS (lpips v0.1, net='vgg') trunk: VGG-16 features[0:30] under lpips.LPIPS().state_dict() names.  conv1_1 is a 1x1
// convolution over the im2col input (27 of 64 columns) that the packer forms from the scaled input, because the zero
// padding of the convolution belongs to the scaled space.  Every convolution has its dgrad twin.
constexpr int kVggStages = 5;
constexpr int kVggConvs[kVggStages] = {2, 2, 3, 3, 3};
constexpr int kVggWidth[kVggStages] = {64, 128, 256, 512, 512};

int build_model_lpips(b2e_unet* m) {
  const int PL = m->PL;
  m->in_im2col = true;
  int idx = 0, cin = 3, n = 0;
  for (int s = 0; s < kVggStages; ++s) {
    for (int j = 0; j < kVggConvs[s]; ++j, ++n) {
      const std::string name = "net.slice" + std::to_string(s + 1) + "." + std::to_string(idx);
      const int cout = kVggWidth[s];
      if (n == 0) {
        ConvL ci;
        ci.cin = ci.cin_pad = kConvBlockK; ci.cout = cout; ci.k = 1; ci.cout_pad = conv_cout_pad(cout); ci.row_len = kConvBlockK * PL;
        ci.w = m->dmalloc<f16>((size_t)ci.cout_pad * ci.row_len);
        ci.b = m->dmalloc<float>(ci.cout_pad);
        ci.dg = m->make_dgrad(kConvBlockK, ci.cout_pad, 1);   // gradient w.r.t. the 64 im2col columns
        const ConvL cd = m->dgrads[ci.dg];
        m->add_param(name + ".weight", (int64_t)cout * 27, 27, [ci, cd, PL](const float* src, cudaStream_t st) {
          const float ws = PL == 3 ? b2e_unet::kSplitWScale : 1.f;
          int rc = conv_pack_weight(src, ci.w, ci.cout, 3, 3, 3, ci.row_len, 0, st, 0, 0, 0, ws);
          if (!rc && PL == 3) rc = conv_pack_weight(src, ci.w, ci.cout, 3, 3, 3, ci.row_len, kConvBlockK, st, 0, 0, 0, ws);
          if (!rc && PL == 3) rc = conv_pack_weight(src, ci.w, ci.cout, 3, 3, 3, ci.row_len, 2 * kConvBlockK, st, 0, 0, 1, ws);
          if (!rc) rc = conv_pack_weight_im2col_T(src, cd.w, ci.cout, 3, cd.row_len, st);
          return rc;
        });
        m->add_f32(name + ".bias", ci.b, cout, 27);
        m->vgg.push_back(ci);
      } else {
        m->vgg.push_back(m->make_conv(name, cin, cout, 3));
      }
      cin = cout;
      idx += 2;                  // conv, ReLU
    }
    idx += 1;                    // max pool
  }
  for (int k = 0; k < kVggStages; ++k) {
    m->lin_w[k] = m->dmalloc<float>(kVggWidth[k]);
    m->add_f32("lin" + std::to_string(k) + ".model.1.weight", m->lin_w[k], kVggWidth[k], kVggWidth[k]);
  }
  const float shift[3] = {-.030f, -.088f, -.188f}, scale[3] = {.458f, .448f, .450f};
  float c[15] = {};
  for (int i = 0; i < 3; ++i) { c[i] = shift[i]; c[3 + i] = scale[i]; c[6 + 4 * i] = 1.f / scale[i]; }
  m->lp_const = m->dmalloc<float>(15);
  if (m->lp_const && cudaMemcpy(m->lp_const, c, sizeof(c), cudaMemcpyHostToDevice) != cudaSuccess) m->build_error = B2E_CUDA_ERROR;
  return m->build_error;
}

// Launch lists of the LPIPS network for batch B.  Forward: input packing (1 - mask * x, scaling layer, im2col) -> VGG
// trunk -> one head launch per tap -> fixed-order final sum.  In reference mode (b2e_lpips_set_reference) the same list
// writes the normalised tap features to the cache instead.  Backward: head gradients joined tap by tap (relu5_3 ->
// relu1_2) into the dgrad chain, max-pool backward, im2col / scaling-layer / mask adjoint.
int build_program_lpips(b2e_unet* m, int B, void* ws, size_t ws_bytes, size_t* need) {
  Arena ar;
  ar.reset(ws, ws_bytes);
  const bool dry = ar.dry;
  std::vector<b2e_unet::Op> fwd, bwd;
  std::vector<b2e_unet::Op>* cur = &fwd;
  double flops = 0;
  int rc = B2E_OK;
  const int PL = m->PL, S = m->lcfg.input_size;
  int tap_hw[kVggStages];
  for (int k = 0; k < kVggStages; ++k) tap_hw[k] = (S >> k) * (S >> k);
  // the reference cache comes first, sized for max_batch: same offset for every batch the program is rebuilt for
  size_t ref_floats = 0;
  for (int k = 0; k < kVggStages; ++k) { m->lp_ref_off[k] = ref_floats; ref_floats += (size_t)m->max_batch * tap_hw[k] * kVggWidth[k]; }
  float* ref = (float*)ar.alloc(ref_floats * sizeof(float));
  auto talloc = [&](int N, int H, int W, int C, int planes = 1) {
    Tensor t; t.N = N; t.H = H; t.W = W; t.C = C; t.Cr = C; t.bytes = (size_t)N * H * W * C * planes * sizeof(f16);
    t.p = (f16*)ar.alloc(t.bytes);
    return t;
  };
  const size_t split_bytes = (size_t)kNumSMs * kConvBlockM * 128 * sizeof(float);
  float* split_ws = (float*)ar.alloc(split_bytes);
  int* split_cnt = (int*)ar.alloc(sizeof(int) * 1024);
  if (!dry) cudaMemset(split_cnt, 0, sizeof(int) * 1024);
  LpipsTaps taps{};
  int nslots = 0;
  for (int k = 0; k < kVggStages; ++k) { taps.n[k] = lpips_head_blocks(tap_hw[k]); taps.off[k] = nslots; taps.hw[k] = tap_hw[k]; nslots += taps.n[k]; }
  double* partial = (double*)ar.alloc(sizeof(double) * B * nslots);
  float* hmax = (float*)ar.alloc(sizeof(float) * B);      // largest head-gradient element per image (gradient scale)
  auto conv = [&](const ConvL& L, const Tensor& x, Tensor* out, const char* what) {
    if (rc) return;
    *out = talloc(B, x.H, x.W, L.cout_pad, PL);
    flops += 2.0 * B * x.H * x.W * (double)L.cout_pad * L.k * L.k * x.C * PL;
    if (dry) return;
    if (PL * L.k * L.k * x.C != L.row_len) {
      rc = B2E_INVALID_ARG; set_error("lpips: operand widths do not match the packed weights (%s)", what); return;
    }
    ConvDesc d;
    d.s0 = ConvSrc{x.p, x.C * PL};
    d.out_planes = PL;
    d.N = B; d.H = x.H; d.W = x.W; d.ksize = L.k; d.stride = 1;
    d.w_packed = L.w; d.Cout = L.cout_pad; d.out_f16 = out->p;
    d.split_ws = split_ws; d.split_ws_bytes = split_bytes; d.split_counters = split_cnt;
    ConvPlan pl;
    rc = conv_plan_build(&pl, d);
    if (rc) return;
    ConvEpilogue ep;
    ep.bias = L.b; ep.relu = 1;
    if (PL == 3) ep.acc_scale = 1.f / b2e_unet::kSplitWScale;
    char desc[160];
    snprintf(desc, sizeof(desc), "%s: conv%dx%d %dx%d cin%d cout%d bn%d%s +relu", what, L.k, L.k, x.H, x.W, x.C, L.cout, pl.block_n,
             pl.halo ? " halo" : pl.pair ? " pair" : "");
    cur->push_back({[pl, ep](cudaStream_t st) { return conv_launch(pl, ep, st); }, 0, pl.flops, 0.0, desc});
  };
  auto ew = [&](std::function<int(cudaStream_t)> fn, double bytes, const char* what) {
    if (!dry && !rc) cur->push_back({std::move(fn), 3, 0.0, bytes, what});
  };

  // ---------------- forward
  ew([hmax, B](cudaStream_t st) -> int { B2E_CUDA(cudaMemsetAsync(hmax, 0, sizeof(float) * B, st)); return (int)B2E_OK; }, 4.0 * B,
     "lpips: clear the head-gradient bound");
  Tensor cols = talloc(B, S, S, kConvBlockK, PL);
  ew([m, cols, B, S, PL](cudaStream_t st) {
       return pack_input_launch(m->in_x, cols.p, B, 3, S, S, kConvBlockK, true, st, PL, nullptr, m->lp_const, m->lp_const + 3,
                                m->lp_mask, m->lp_mask_batched); },
     (double)B * S * S * 12.0 + (double)cols.bytes, "input: 1 - mask * x, scaling layer, im2col");
  std::vector<Tensor> acts(m->vgg.size());
  Tensor tap[kVggStages], h = cols;
  uint16_t* pidx[kVggStages] = {};
  int li = 0;
  for (int s = 0; s < kVggStages && !rc; ++s) {
    if (s > 0) {
      Tensor p = talloc(B, h.H / 2, h.W / 2, h.C, PL);
      pidx[s - 1] = (uint16_t*)ar.alloc(sizeof(uint16_t) * (size_t)B * p.H * p.W * (p.C / 8));
      const Tensor hh = h;
      uint16_t* ix = pidx[s - 1];
      ew([hh, p, ix, B, PL](cudaStream_t st) { return maxpool2x2_launch(hh.p, p.p, ix, B, hh.H, hh.W, hh.C, st, PL); },
         1.25 * (double)hh.bytes, "maxpool 2x2");
      h = p;
    }
    for (int j = 0; j < kVggConvs[s]; ++j, ++li) {
      conv(m->vgg[li], h, &acts[li], "vgg");
      h = acts[li];
    }
    tap[s] = h;
  }
  for (int k = 0; k < kVggStages && !rc; ++k) {
    const Tensor t = tap[k];
    const int slot0 = taps.off[k];
    float* rk = ref + m->lp_ref_off[k];
    ew([m, t, k, rk, partial, nslots, slot0, hmax, B, PL](cudaStream_t st) {
         const bool rmode = m->lp_ref_mode;
         return lpips_head_launch(t.p, B, t.C, t.H * t.W, PL, m->lin_w[k], rk, rmode ? 0 : m->lp_ref_B != 1, partial, nslots, slot0,
                                  rmode ? 0 : 1, hmax, st); },
       (double)t.bytes + 4.0 * B * t.H * t.W * t.C, "lpips head (normalise, lin, spatial sum)");
  }
  ew([m, partial, nslots, taps, B](cudaStream_t st) {
       return m->lp_ref_mode ? (int)B2E_OK : lpips_finalize_launch(partial, nslots, taps, m->out_eps, B, st); },
     8.0 * B * nslots, "lpips: sum over taps");

  // ---------------- backward: d(dist) -> d(input)
  if (!rc && m->grad) {
    cur = &bwd;
    auto dconv = [&](const ConvL& L, const Tensor& dy, Tensor* dx) {
      if (rc) return;
      const ConvL& D = m->dgrads[L.dg];
      *dx = talloc(B, dy.H, dy.W, D.cout_pad);
      flops += 2.0 * B * dy.H * dy.W * (double)D.cout_pad * D.row_len;
      if (dry) return;
      if (D.k * D.k * dy.C != D.row_len) { rc = B2E_INVALID_ARG; set_error("lpips backward: operand widths do not match"); return; }
      ConvDesc d;
      d.s0 = ConvSrc{dy.p, dy.C};
      d.N = B; d.H = dy.H; d.W = dy.W; d.ksize = D.k; d.stride = 1;
      d.w_packed = D.w; d.Cout = D.cout_pad; d.out_f16 = dx->p;
      d.split_ws = split_ws; d.split_ws_bytes = split_bytes; d.split_counters = split_cnt;
      ConvPlan pl;
      rc = conv_plan_build(&pl, d);
      if (rc) return;
      char desc[160];
      snprintf(desc, sizeof(desc), "vgg: dgrad conv%dx%d %dx%d cin%d cout%d", D.k, D.k, dy.H, dy.W, dy.C, D.cout);
      cur->push_back({[pl](cudaStream_t st) { return conv_launch(pl, ConvEpilogue{}, st); }, 0, pl.flops, 0.0, desc});
    };
    // gradient scale record (grad_scale_launch) from the largest head-gradient element the forward measured (it includes
    // the 1 / ||f|| of the normalisation Jacobian, so the scale follows the feature norms of the actual weights)
    float* gsc = (float*)ar.alloc(sizeof(float) * 4);
    float* gprod = (float*)ar.alloc(sizeof(float) * B);
    if (!dry) cudaMemset(gsc, 0, sizeof(float) * 4);
    ew([m, hmax, gprod, gsc, B](cudaStream_t st) { return lpips_grad_scale_launch(m->in_dlogits, hmax, gprod, B, gsc, st); },
       8.0 * B, "max |d(dist)| x head-gradient bound -> power-of-two gradient scale");
    Tensor gp;      // gradient arriving at the current tap through the max pool above it (none at relu5_3)
    li = (int)m->vgg.size() - 1;
    for (int s = kVggStages - 1; s >= 0 && !rc; --s) {
      const Tensor t = tap[s];
      Tensor g = talloc(B, t.H, t.W, t.C);
      const f16* gpp = s == kVggStages - 1 ? nullptr : gp.p;
      float* rk = ref + m->lp_ref_off[s];
      ew([m, t, s, rk, gsc, gpp, g, B, PL](cudaStream_t st) {
           return lpips_head_bwd_launch(t.p, B, t.C, t.H * t.W, PL, m->lin_w[s], rk, m->lp_ref_B != 1, m->in_dlogits, gsc, gpp, g.p, st); },
         (double)t.bytes + 4.0 * B * t.H * t.W * t.C + 2.0 * (double)g.bytes, "lpips head backward (+ pooled path, relu mask)");
      for (int j = kVggConvs[s] - 1; j >= 0 && !rc; --j, --li) {
        Tensor dx;
        dconv(m->vgg[li], g, &dx);
        if (j > 0) {
          const Tensor gg = dx, yy = acts[li - 1];
          ew([gg, yy, PL](cudaStream_t st) { return relu_bwd_launch(gg.p, yy.p, gg.p, (int64_t)(gg.bytes / sizeof(f16)), st, PL, gg.C); },
             3.0 * (double)gg.bytes, "relu backward");
        }
        g = dx;
      }
      if (rc) break;
      if (s > 0) {
        // g = d(pool output): to the arg-max positions of the tap below (+ its ReLU mask)
        const Tensor tb = tap[s - 1], gy = g;
        gp = talloc(B, tb.H, tb.W, tb.C);
        const Tensor gx = gp;
        uint16_t* ix = pidx[s - 1];
        ew([tb, ix, gy, gx, B, PL](cudaStream_t st) { return maxpool2x2_bwd_launch(tb.p, ix, gy.p, gx.p, B, tb.H, tb.W, tb.C, st, PL); },
           2.5 * (double)gx.bytes, "maxpool 2x2 backward (+ relu mask)");
      } else {
        const Tensor dc = g;
        ew([m, dc, gsc, B, S](cudaStream_t st) {
             return vq_col2im_bwd_launch(dc.p, m->lp_const + 6, m->out_dz, B, 3, S, S, st, gsc, m->lp_mask, m->lp_mask_batched); },
           (double)dc.bytes + 12.0 * B * S * S, "col2im + scaling layer + input mask backward");
      }
    }
    cur = &fwd;
  }
  if (rc) return rc;
  if (need) *need = ar.peak;
  if (!dry) {
    B2E_REQUIRE(ar.peak <= ws_bytes, B2E_WORKSPACE_TOO_SMALL, "lpips: workspace too small (%zu > %zu)", ar.peak, ws_bytes);
    m->ops = std::move(fwd);
    m->bops = std::move(bwd);
    m->fwd_B = -1;
    m->cur_B = B;
  }
  m->flops = flops;
  return B2E_OK;
}

int build_model_clip(b2e_unet* m) {
  const b2e_clip_config& c = m->ccfg;
  const int D = c.hidden_size;
  m->tok_emb = m->dmalloc<float>((size_t)c.vocab_size * D);
  m->pos_emb = m->dmalloc<float>((size_t)c.max_positions * D);
  m->add_f32("text_model.embeddings.token_embedding.weight", m->tok_emb, (int64_t)c.vocab_size * D, -50);
  m->add_f32("text_model.embeddings.position_embedding.weight", m->pos_emb, (int64_t)c.max_positions * D, -50);
  for (int i = 0; i < c.num_layers; ++i) {
    const std::string b = "text_model.encoder.layers." + std::to_string(i);
    b2e_unet::ClipL L;
    L.ln1 = m->make_ln(b + ".layer_norm1", D);
    L.qkv = m->make_fused_linear(b + ".self_attn", {"q_proj", "k_proj", "v_proj"}, D, D, true);
    L.out = m->make_linear(b + ".self_attn.out_proj", D, D, true, D);
    L.ln2 = m->make_ln(b + ".layer_norm2", D);
    L.fc1 = m->make_linear(b + ".mlp.fc1", D, c.intermediate_size, true);
    L.fc2 = m->make_linear(b + ".mlp.fc2", c.intermediate_size, D, true, D);
    m->clayers.push_back(L);
  }
  m->clip_final_ln = m->make_ln("text_model.final_layer_norm", D);
  return m->build_error;
}

int build_model(b2e_unet* m) {
  if (m->clip) return build_model_clip(m);
  if (m->resnet) return build_model_resnet(m);
  if (m->lpips) return build_model_lpips(m);
  if (m->decoder) return build_model_decoder(m);
  if (m->encoder) return build_model_encoder(m);
  const b2e_unet_config& c = m->cfg;
  const int nb = c.n_blocks;
  const int c0 = c.block_out_channels[0];
  m->temb_dim = 4 * c0;
  // conv_in: with <= 7 input channels the 9 taps x Cin values of a pixel fit ONE 64-channel K chunk, so the input
  // is packed as an im2col tensor (B,S,S,64) and conv_in runs as a 1x1 convolution (1 k-block instead of 9)
  m->in_im2col = c.in_channels == 1 || c.in_channels == 3 || c.in_channels == 4;
  if (m->in_im2col) {
    ConvL ci;
    const int PL = m->PL;
    ci.cin = ci.cin_pad = kConvBlockK; ci.cout = c0; ci.k = 1; ci.cout_pad = conv_cout_pad(c0); ci.row_len = kConvBlockK * PL;
    ci.w = m->dmalloc<f16>((size_t)ci.cout_pad * ci.row_len);
    ci.b = m->dmalloc<float>(ci.cout_pad);
    const int cin = c.in_channels;
    m->add_param("conv_in.weight", (int64_t)c0 * cin * 9, (int64_t)cin * 9, [ci, cin, PL](const float* src, cudaStream_t st) {
      // column of (tap t, channel c) = t * Cin + c, the order pack_input_im2col writes (per 64-column plane)
      const float ws = PL == 3 ? b2e_unet::kSplitWScale : 1.f;
      int rc = conv_pack_weight(src, ci.w, ci.cout, cin, 3, cin, ci.row_len, 0, st, 0, 0, 0, ws);
      if (!rc && PL == 3) rc = conv_pack_weight(src, ci.w, ci.cout, cin, 3, cin, ci.row_len, kConvBlockK, st, 0, 0, 0, ws);
      if (!rc && PL == 3) rc = conv_pack_weight(src, ci.w, ci.cout, cin, 3, cin, ci.row_len, 2 * kConvBlockK, st, 0, 0, 1, ws);
      return rc;
    });
    m->add_f32("conv_in.bias", ci.b, c0, (int64_t)cin * 9);
    m->conv_in = ci;
  } else {
    m->conv_in = m->make_conv("conv_in", c.in_channels, c0, 3, kConvBlockK);
  }
  m->te_w1 = m->dmalloc<float>((size_t)m->temb_dim * c0); m->te_b1 = m->dmalloc<float>(m->temb_dim);
  m->te_w2 = m->dmalloc<float>((size_t)m->temb_dim * m->temb_dim); m->te_b2 = m->dmalloc<float>(m->temb_dim);
  m->add_f32("time_embedding.linear_1.weight", m->te_w1, (int64_t)m->temb_dim * c0, c0);
  m->add_f32("time_embedding.linear_1.bias", m->te_b1, m->temb_dim, c0);
  m->add_f32("time_embedding.linear_2.weight", m->te_w2, (int64_t)m->temb_dim * m->temb_dim, m->temb_dim);
  m->add_f32("time_embedding.linear_2.bias", m->te_b2, m->temb_dim, m->temb_dim);
  std::vector<int> stack;  // channel counts of the skip stack
  stack.push_back(c0);
  m->nodes.push_back({N_PUSH, 0});
  int ch = c0;
  for (int i = 0; i < nb; ++i) {
    const int cout = c.block_out_channels[i];
    for (int j = 0; j < c.layers_per_block; ++j) {
      const std::string base = "down_blocks." + std::to_string(i);
      m->nodes.push_back({N_RESNET, m->make_resnet(base + ".resnets." + std::to_string(j), ch, 0, cout)});
      ch = cout;
      if (c.down_attn[i]) {
        if (c.cross_attention_dim > 0)
          m->nodes.push_back({N_XFORMER, m->make_xformer(base + ".attentions." + std::to_string(j), ch, c.num_attention_heads, c.cross_attention_dim)});
        else
          m->nodes.push_back({N_ATTN, m->make_attn(base + ".attentions." + std::to_string(j), ch)});
      }
      m->nodes.push_back({N_PUSH, 0});
      stack.push_back(ch);
    }
    if (i != nb - 1) {
      m->downs.push_back(m->make_conv("down_blocks." + std::to_string(i) + ".downsamplers.0.conv", ch, ch, 3));
      m->nodes.push_back({N_DOWN, (int)m->downs.size() - 1});
      m->nodes.push_back({N_PUSH, 0});
      stack.push_back(ch);
    }
  }
  m->nodes.push_back({N_RESNET, m->make_resnet("mid_block.resnets.0", ch, 0, ch)});
  if (c.cross_attention_dim > 0)
    m->nodes.push_back({N_XFORMER, m->make_xformer("mid_block.attentions.0", ch, c.num_attention_heads, c.cross_attention_dim)});
  else
    m->nodes.push_back({N_ATTN, m->make_attn("mid_block.attentions.0", ch)});
  m->nodes.push_back({N_RESNET, m->make_resnet("mid_block.resnets.1", ch, 0, ch)});
  for (int i = 0; i < nb; ++i) {
    const int cout = c.block_out_channels[nb - 1 - i];
    const std::string base = "up_blocks." + std::to_string(i);
    for (int j = 0; j < c.layers_per_block + 1; ++j) {
      const int skip = stack.back();
      stack.pop_back();
      m->nodes.push_back({N_POPCAT, 0});
      m->nodes.push_back({N_RESNET, m->make_resnet(base + ".resnets." + std::to_string(j), ch, skip, cout)});
      ch = cout;
      if (c.up_attn[i]) {
        if (c.cross_attention_dim > 0)
          m->nodes.push_back({N_XFORMER, m->make_xformer(base + ".attentions." + std::to_string(j), ch, c.num_attention_heads, c.cross_attention_dim)});
        else
          m->nodes.push_back({N_ATTN, m->make_attn(base + ".attentions." + std::to_string(j), ch)});
      }
    }
    if (i != nb - 1) {
      m->ups.push_back(m->make_conv(base + ".upsamplers.0.conv", ch, ch, 3, 0, 0, 0, true));
      m->nodes.push_back({N_UP, (int)m->ups.size() - 1});
    }
  }
  B2E_REQUIRE(stack.empty(), B2E_INVALID_ARG, "unet: skip stack not empty (%zu left)", stack.size());
  m->norm_out = m->make_norm("conv_norm_out", ch);
  m->conv_out = m->make_conv("conv_out", ch, c.out_channels, 3);
  // all time_emb_proj layers as one [sumC][temb_dim] matrix
  m->tp_w = m->dmalloc<float>((size_t)m->sumC * m->temb_dim);
  m->tp_b = m->dmalloc<float>(m->sumC);
  for (auto& r : m->resnets) {
    m->add_f32(r.name + ".time_emb_proj.weight", m->tp_w + (size_t)r.temb_off * m->temb_dim,
               (int64_t)r.cout * m->temb_dim, m->temb_dim);
    m->add_f32(r.name + ".time_emb_proj.bias", m->tp_b + r.temb_off, r.cout, m->temb_dim);
  }
  return m->build_error;
}

// installs a forward-only launch list (text encoder)
int finish_forward_only(b2e_unet* m, std::vector<b2e_unet::Op>& fwd, size_t peak, size_t ws_bytes, size_t* need, bool dry,
                        double flops, int B) {
  if (need) *need = peak;
  if (!dry) {
    B2E_REQUIRE(peak <= ws_bytes, B2E_WORKSPACE_TOO_SMALL, "text encoder: workspace too small (%zu > %zu)", peak, ws_bytes);
    m->ops = std::move(fwd);
    m->bops.clear();
    m->fwd_B = -1;
    m->cur_B = B;
  }
  m->flops = flops;
  return B2E_OK;
}

// Records the launch list for batch B with all activations placed in the arena.  With a null
// arena base this is a dry run that only measures the arena size.
int build_program(b2e_unet* m, int B, void* ws, size_t ws_bytes, size_t* need) {
  if (m->resnet) return build_program_resnet(m, B, ws, ws_bytes, need);
  if (m->lpips) return build_program_lpips(m, B, ws, ws_bytes, need);
  const b2e_unet_config& c = m->cfg;
  Arena ar;
  ar.reset(ws, ws_bytes);
  const bool dry = ar.dry;
  std::vector<b2e_unet::Op> ops_fwd, ops_bwd;
  std::vector<b2e_unet::Op>* cur = &ops_fwd;   // the op list being recorded
#define ops (*cur)
  const bool keep = m->grad;                    // gradient mode: every activation stays live for the backward pass
  const int PL = m->PL;                         // channel planes per activation tensor (3: split-f16, fp32-accurate mode)
  double flops = 0;
  int rc = B2E_OK;
  auto talloc = [&](int N, int H, int W, int C, int Cr = 0) {
    Tensor t; t.N = N; t.H = H; t.W = W; t.C = C; t.Cr = Cr ? Cr : C; t.bytes = (size_t)N * H * W * C * PL * sizeof(f16);
    t.p = (f16*)ar.alloc(t.bytes);
    return t;
  };
  auto tfree = [&](Tensor& t) {
    if (t.alias) {   // a fused-GroupNorm view owns only its coefficient table
      if (t.gn_coef && !keep) ar.release(t.gn_coef, sizeof(float) * 2 * (size_t)t.N * t.C);
      t.gn_coef = nullptr; t.p = nullptr;
      return;
    }
    if (keep) return;
    if (t.p) ar.release(t.p, t.bytes);
    if (t.cstats) ar.release(t.cstats, sizeof(float) * 2 * t.N * t.C);
    if (t.tstats) ar.release(t.tstats, t.tstats_bytes);
    t.p = nullptr; t.cstats = nullptr; t.tstats = nullptr;
  };
  const int G = c.norm_num_groups;
  const int S = c.sample_size;
  // per-forward scratch
  float* act = (float*)ar.alloc(sizeof(float) * B * (m->temb_dim > 0 ? m->temb_dim : 1));
  float* proj = (float*)ar.alloc(sizeof(float) * B * (m->sumC > 0 ? m->sumC : 1));
  float* gn_part = (float*)ar.alloc(sizeof(float) * B * 64 * G * 2);
  // split-K scratch for the low-resolution convolutions (<= one 128x128 fp32 partial tile per SM) + tile counters
  const size_t split_bytes = (size_t)kNumSMs * kConvBlockM * 128 * sizeof(float);
  float* split_ws = (float*)ar.alloc(split_bytes);
  int* split_cnt = (int*)ar.alloc(sizeof(int) * 1024);
  if (!dry) cudaMemset(split_cnt, 0, sizeof(int) * 1024);

  auto conv = [&](const ConvL& L, Tensor x0, const Tensor* x1, int stride, ConvEpilogue ep, Tensor* out, float* out_nchw,
                  const Tensor* r0 = nullptr, const Tensor* r1 = nullptr, bool want_stats = true) {
    if (rc) return;
    const int Ho = x0.H / stride, Wo = x0.W / stride;
    // f16 outputs are written at the padded channel count (zero weight rows / bias for the tail)
    const int cout_x = out ? L.cout_pad : L.cout;
    if (out) *out = talloc(B, Ho, Wo, cout_x, L.cout);
    // GroupNorm statistics of the output, emitted by the epilogue (the consumer skips its statistics pass)
    const ConvGeom geo = conv_geometry(B, Ho, Wo, cout_x, L.k, stride);
    float* tstats = nullptr;
    const size_t tstats_bytes = sizeof(float) * 2 * (size_t)conv_stats_slots(geo) * cout_x;
    // few tile slots per image (low-resolution levels): the consumer reduces them itself
    const bool raw_stats = geo.w_blks * geo.h_blks <= 16;
    if (out && want_stats && geo.stats_ok && PL == 1) {
      tstats = (float*)ar.alloc(tstats_bytes);
      if (raw_stats) {
        out->tstats = tstats; out->tstats_bytes = tstats_bytes; out->ts_nt = geo.Nt; out->ts_per_img = geo.w_blks * geo.h_blks;
      } else {
        out->cstats = (float*)ar.alloc(sizeof(float) * 2 * B * cout_x);
      }
    }
    if (dry) {
      flops += 2.0 * B * Ho * Wo * (double)cout_x * (L.k * L.k * (x0.C + (x1 ? x1->C : 0)) + L.res_c) * PL;
      if (tstats && !raw_stats) ar.release(tstats, tstats_bytes);
      return;
    }
    ConvDesc d;
    d.s0 = ConvSrc{x0.p, x0.C * PL};
    if (x1) d.s1 = ConvSrc{x1->p, x1->C * PL};
    if (x0.alias) {
      if (x1 || stride != 1) { rc = B2E_INVALID_ARG; set_error("unet: fused GroupNorm view used as a second source / strided input"); return; }
      d.s0 = ConvSrc{x0.p, x0.C0};
      if (x0.p1) d.s1 = ConvSrc{x0.p1, x0.C1};
      d.gn_coef = x0.gn_coef; d.gn_silu = x0.gn_silu;
    }
    if (r0) d.r0 = ConvSrc{r0->p, r0->C * PL};
    if (r1) d.r1 = ConvSrc{r1->p, r1->C * PL};
    d.out_planes = out ? PL : 1;
    d.N = B; d.H = x0.H; d.W = x0.W; d.ksize = L.k; d.stride = stride; d.w_packed = L.w; d.Cout = cout_x;
    d.stride2_pad1 = c.downsample_padding == 1;
    if (PL * (L.k * L.k * (x0.C + (x1 ? x1->C : 0)) + L.res_c) != L.row_len) {
      rc = B2E_INVALID_ARG; set_error("unet: weight row length %d does not match the operands (%d)", L.row_len,
                                      PL * (L.k * L.k * (x0.C + (x1 ? x1->C : 0)) + L.res_c)); return;
    }
    d.out_f16 = out ? out->p : nullptr;
    d.tile_stats = tstats;
    d.split_ws = split_ws; d.split_ws_bytes = split_bytes; d.split_counters = split_cnt;
    if (L.res_c != (r0 ? r0->C : 0) + (r1 ? r1->C : 0)) { rc = B2E_INVALID_ARG; set_error("unet: residual segment mismatch"); return; }
    ConvPlan pl;
    rc = conv_plan_build(&pl, d);
    if (rc) return;
    ep.bias = L.b;
    ep.bias2 = L.b2;
    if (PL == 3) ep.acc_scale = 1.f / b2e_unet::kSplitWScale;
    flops += pl.flops;
    char desc[160];
    snprintf(desc, sizeof(desc), "conv%dx%d s%d %dx%d cin%d+%d res%d cout%d tiles%d bn%d%s", L.k, L.k, stride, x0.H, x0.W,
             x0.C, x1 ? x1->C : 0, L.res_c, L.cout, pl.w_blks * pl.h_blks * pl.n_blks * (pl.cout_pad / pl.block_n), pl.block_n,
             pl.halo == 2 ? " halo2" : pl.halo ? " halo1" : pl.pair ? " pair" : (pl.splits > 1 ? ((pl.split_cluster ? " clusterK" : " splitK") + std::to_string(pl.splits)).c_str() : ""));
    if (x0.alias) snprintf(desc + strlen(desc), sizeof(desc) - strlen(desc), " +gn%s", x0.gn_silu ? "+silu" : "");
    // profile record: ALGORITHMIC FLOPs.  An identity residual segment (W_r = I: the plain residual add riding along as
    // K chunks) is executed on the tensor cores but is not arithmetic of the algorithm - it is counted as the bytes of the
    // residual tensor it reads instead (conv_shortcut segments, which have a bias2, are real 1x1 convolutions and count)
    const bool id_res = L.res_c > 0 && !L.b2;
    const double id_flops = id_res ? 2.0 * B * Ho * Wo * (double)cout_x * L.res_c * PL : 0.0;
    const double id_bytes = id_res ? (double)B * Ho * Wo * L.res_c * PL * sizeof(f16) : 0.0;
    if (out_nchw) {
      // the network output pointer is only known at call time
      ops.push_back({[pl, ep, m](cudaStream_t st) { ConvEpilogue e = ep; e.out_f32_nchw = m->out_eps; return conv_launch(pl, e, st); },
                     0, pl.flops - id_flops, id_bytes, desc});
    } else {
      ops.push_back({[pl, ep](cudaStream_t st) { return conv_launch(pl, ep, st); }, 0, pl.flops - id_flops, id_bytes, desc});
    }
    if (tstats && !raw_stats) {
      float* cst = out->cstats;
      const int C = cout_x;
      const int fNt = pl.Nt, fw = pl.w_blks, fh = pl.h_blks;   // the plan's actual tiling (halo mode re-tiles)
      ops.push_back({[tstats, cst, B, C, fNt, fw, fh](cudaStream_t st) {
                       return gn_finalize_launch(tstats, cst, B, C, fNt, fw, fh, st);
                     }, 3, 0.0, (double)tstats_bytes});
      ar.release(tstats, tstats_bytes);   // dead after the finalize kernel (stream order)
    }
  };
  // Upsampler: nearest x2 followed by a 3x3 convolution, computed as FOUR 2x2 convolutions over the low-resolution tensor
  // (one per output-pixel parity, weights pre-summed at set_param time): 2.25x fewer FLOPs, and the upsampled tensor is
  // never written or read.  Each phase writes its sub-grid of the output through a strided TMA map and its own block of
  // GroupNorm tile statistics; ONE gn_finalize reduces the four blocks.  Forward-only programs, outputs of >= 128x128.
  // Measured at batch 8 (DDPM-256, tools/profile_ops.py): 128 -> 256 at 128 channels 4 x 29.2 us against 115 us + 52 us of
  // upsample2x; 64 -> 128 at 256 channels 4 x 24.6 against 98 + 29; 32 -> 64 at 256 channels 4 x 15 against 36 + 15 (worse:
  // excluded).  The phase launches are K-short (8-16 k-blocks per tile) and therefore epilogue-bound at 580-700 TFLOP/s:
  // the gain is the upsample pass they remove, not their 2.25x fewer FLOPs.  B2E_UP2=0 restores upsample2x + conv3x3.
  static const bool up2_on = !(getenv("B2E_UP2") && atoi(getenv("B2E_UP2")) == 0);
  auto conv_up2 = [&](const ConvL& L, const Tensor& x, Tensor* out) {
    if (rc) return;
    const int cout_x = L.cout_pad;
    *out = talloc(B, 2 * x.H, 2 * x.W, cout_x, L.cout);
    const ConvGeom geo = conv_geometry(B, x.H, x.W, cout_x, 2, 1);     // tiling of ONE phase (the low-resolution grid)
    const size_t slots = (size_t)conv_stats_slots(geo);
    const size_t tstats_bytes = sizeof(float) * 2 * 4 * slots * cout_x;
    float* tstats = nullptr;
    if (geo.stats_ok && PL == 1) {
      tstats = (float*)ar.alloc(tstats_bytes);
      out->cstats = (float*)ar.alloc(sizeof(float) * 2 * B * cout_x);
    }
    const double fl = 4 * 2.0 * B * x.H * x.W * (double)cout_x * (4.0 * x.C) * PL;
    if (dry) {
      flops += fl;
      if (tstats) ar.release(tstats, tstats_bytes);
      return;
    }
    if (PL * 4 * x.C != L.row_len_up2) { rc = B2E_INVALID_ARG; set_error("unet: upsampler operand width does not match the packed phase weights"); return; }
    int fNt = geo.Nt, fw = geo.w_blks, fh = geo.h_blks;
    for (int ph = 0; ph < 4 && !rc; ++ph) {
      ConvDesc d;
      d.s0 = ConvSrc{x.p, x.C * PL};
      d.out_planes = PL;
      d.N = B; d.H = x.H; d.W = x.W; d.ksize = 2; d.stride = 1; d.up2_phase = ph;
      d.w_packed = L.w_up2 + (size_t)ph * L.cout_pad * L.row_len_up2; d.Cout = cout_x; d.out_f16 = out->p;
      d.tile_stats = tstats ? tstats + (size_t)ph * slots * cout_x * 2 : nullptr;
      d.split_ws = split_ws; d.split_ws_bytes = split_bytes; d.split_counters = split_cnt;
      ConvPlan pl;
      rc = conv_plan_build(&pl, d);
      if (rc) return;
      ConvEpilogue ep;
      ep.bias = L.b;
      if (PL == 3) ep.acc_scale = 1.f / b2e_unet::kSplitWScale;
      flops += pl.flops;
      fNt = pl.Nt; fw = pl.w_blks; fh = pl.h_blks;
      char desc[160];
      snprintf(desc, sizeof(desc), "upsample x2 + conv3x3 as 2x2 phase %d: %dx%d -> %dx%d cin%d cout%d tiles%d bn%d%s", ph, x.H, x.W,
               2 * x.H, 2 * x.W, x.C, L.cout, pl.w_blks * pl.h_blks * pl.n_blks * (pl.cout_pad / pl.block_n), pl.block_n,
               pl.pair ? " pair" : "");
      ops.push_back({[pl, ep](cudaStream_t st) { return conv_launch(pl, ep, st); }, 0, pl.flops, 0.0, desc});
    }
    if (tstats) {
      float* cst = out->cstats;
      const int C = cout_x;
      const int64_t pstride = (int64_t)slots * cout_x * 2;
      ops.push_back({[tstats, cst, B, C, fNt, fw, fh, pstride](cudaStream_t st) {
                       return gn_finalize_launch(tstats, cst, B, C, fNt, fw, fh, st, 4, pstride);
                     }, 3, 0.0, (double)tstats_bytes});
      ar.release(tstats, tstats_bytes);
    }
  };
  // GroupNorm(+SiLU): statistics come from the producing convolution's epilogue, the apply pass is a stand-alone
  // memory-bound kernel (4 B/elem).  B2E_GN_FUSE=1 (experimental, OFF by default) instead fuses the apply into the consumer
  // convolution (16-bit mode, sources a multiple of 64 channels wide): only the per-(image, channel) coefficients are
  // computed here and *out is a view of the raw source(s); the convolution's transform warps normalise its A operand in
  // shared memory (conv_igemm XF kernels), so the normalised tensor never exists.  Bit-identical results, but measured
  // SLOWER on B200 (profiles/r2_gn_fusion.md): the extra barrier hop per pipeline stage (TMA -> transform warps -> MMA)
  // stalls the 3-4 stage smem ring (+44 % on the 256x256 layers with the transform itself switched off), more than the
  // 1.8 ms of GroupNorm launches it removes.
  static const int gn_fuse_mode = getenv("B2E_GN_FUSE") ? atoi(getenv("B2E_GN_FUSE")) : 0;
  static const bool gn_fuse_on = gn_fuse_mode != 0;
  // B2E_GN_FUSE=<r> with r >= 8: fuse only on feature maps of at most r x r (the latency-bound low-resolution levels)
  const int gn_fuse_max_res = gn_fuse_mode >= 8 ? gn_fuse_mode : (1 << 30);
  auto gnorm = [&](const NormL& L, Tensor x0, const Tensor* x1, int silu, Tensor* out, float** stats_out = nullptr,
                   float eps_override = -1.f) {
    if (rc) return;
    const int C = x0.Cr + (x1 ? x1->Cr : 0);   // real channels, written compactly; pitch rounded up to 64
    const bool fuse = gn_fuse_on && x0.H <= gn_fuse_max_res && PL == 1 && x0.Cr == x0.C && x0.C % kConvBlockK == 0 &&
                      (!x1 || (x1->Cr == x1->C && x1->C % kConvBlockK == 0));
    float* coef = nullptr;
    if (fuse) {
      Tensor t; t.N = B; t.H = x0.H; t.W = x0.W; t.C = C; t.Cr = C; t.bytes = 0;
      t.alias = true; t.p = x0.p; t.C0 = x0.C; t.p1 = x1 ? x1->p : nullptr; t.C1 = x1 ? x1->C : 0; t.gn_silu = silu;
      coef = (float*)ar.alloc(sizeof(float) * 2 * (size_t)B * C);
      t.gn_coef = coef;
      *out = t;
    } else {
      *out = talloc(B, x0.H, x0.W, pad64(C), C);
    }
    float* sv = (keep && stats_out) ? (float*)ar.alloc(sizeof(float) * 2 * B * G) : nullptr;
    if (stats_out) *stats_out = sv;
    if (dry) return;
    GNArgs a;
    a.save_stats = sv;
    a.x0 = x0.p; a.x1 = x1 ? x1->p : nullptr; a.C0 = x0.Cr; a.C1 = x1 ? x1->Cr : 0;
    a.P0 = x0.C; a.P1 = x1 ? x1->C : 0; a.Pout = fuse ? C : out->C;
    a.N = B; a.HW = x0.H * x0.W; a.G = G; a.eps = eps_override > 0.f ? eps_override : c.norm_eps; a.gamma = L.g; a.beta = L.b;
    a.partial = gn_part; a.chunks = gn_chunks(a.HW, C); a.out = fuse ? nullptr : out->p; a.silu = silu; a.planes = PL;
    bool fused = x0.cstats && (!x1 || x1->cstats);
    a.cs0 = fused ? x0.cstats : nullptr;
    a.cs1 = fused && x1 ? x1->cstats : nullptr;
    const bool raw = x0.tstats && (!x1 || (x1->tstats && x1->ts_nt == x0.ts_nt && x1->ts_per_img == x0.ts_per_img));
    a.ts0 = raw ? x0.tstats : nullptr;
    a.ts1 = raw && x1 ? x1->tstats : nullptr;
    a.ts_nt = x0.ts_nt; a.ts_per_img = x0.ts_per_img;
    if (raw) fused = true;
    if (fuse) {
      // algorithmic traffic: the statistics pass reads x only when no producing convolution supplied them
      ops.push_back({[a, coef](cudaStream_t st) { return gn_coeffs_launch(a, coef, st); }, 1, 0.0, (fused ? 0.0 : 2.0) * B * a.HW * C,
                     "groupnorm coefficients (apply fused into the consumer conv)"});
      return;
    }
    // algorithmic traffic: statistics pass reads x, apply pass reads x and writes y (f16)
    ops.push_back({[a](cudaStream_t st) { return gn_launch(a, st); }, 1, 0.0, (fused ? 4.0 : 6.0) * B * a.HW * C});
  };

  // ---- prologue: input packing, timestep embedding
  Tensor xin = talloc(B, S, S, kConvBlockK);
  float* zq = m->decoder ? (float*)ar.alloc(sizeof(float) * B * c.in_channels * S * S) : nullptr;
  if (!dry && !m->clip) {
    const int Cin = c.in_channels, HW = S * S;
    const bool im2col = m->in_im2col;
    if (m->decoder) {
      // latent -> nearest code -> post_quant_conv (fp32 NCHW), then the usual im2col packing of conv_in
      ops.push_back({[m, zq, B, Cin, HW](cudaStream_t st) {
                       return vq_quantize_launch(m->in_x, m->codebook, m->n_codes, m->pq_w, m->pq_b, zq, B, Cin, HW, st);
                     }, 3, 0.0, 8.0 * B * Cin * HW, "vq nearest code + post_quant_conv"});
      ops.push_back({[zq, xin, B, Cin, S, PL](cudaStream_t st) { return pack_input_launch(zq, xin.p, B, Cin, S, S, kConvBlockK, true, st, PL); },
                     3, 0.0, (double)B * HW * (4.0 * Cin + 2.0 * kConvBlockK)});
    } else {
      ops.push_back({[m, xin, B, Cin, S, im2col, PL](cudaStream_t st) { return pack_input_launch(m->in_x, xin.p, B, Cin, S, S, kConvBlockK, im2col, st, PL); },
                     3, 0.0, (double)B * HW * (4.0 * Cin + 2.0 * kConvBlockK)});
    }
    if (!m->decoder && !m->encoder) {
    TembArgs ta;
    ta.timesteps = nullptr; ta.B = B; ta.dim0 = c.block_out_channels[0]; ta.dim = m->temb_dim;
    ta.flip = c.flip_sin_to_cos; ta.freq_shift = c.freq_shift;
    ta.w1 = m->te_w1; ta.b1 = m->te_b1; ta.w2 = m->te_w2; ta.b2 = m->te_b2; ta.wp = m->tp_w; ta.bp = m->tp_b;
    ta.sumC = m->sumC; ta.act = act; ta.proj = proj;
    ops.push_back({[m, ta](cudaStream_t st) { TembArgs t = ta; t.timesteps = m->in_t; return temb_launch(t, st); }, 3, 0.0, 0.0});
    }
  }
  // text conditioning of the conditional UNet: fp32 (B, L <= 128, D) -> f16 (B, 1, 128, D), zero rows beyond L
  constexpr int kCtxPad = 128;
  Tensor ctxp;
  if (c.cross_attention_dim > 0) {
    ctxp = talloc(B, 1, kCtxPad, c.cross_attention_dim);
    if (!dry) {
      const int D = c.cross_attention_dim;
      ops.push_back({[m, ctxp, B, D, PL](cudaStream_t st) { return pack_context_launch(m->in_ctx, ctxp.p, B, m->ctx_len, kCtxPad, D, st, PL); },
                     3, 0.0, (double)B * kCtxPad * D * 6.0, "pack text context"});
    }
  }
  auto lnorm = [&](const LNL& L, const Tensor& x, Tensor* out) {
    if (rc) return;
    *out = talloc(B, x.H, x.W, x.C);
    if (dry) return;
    Tensor xx = x, oo = *out;
    const int64_t rows = (int64_t)B * x.H * x.W;
    ops.push_back({[L, xx, oo, rows, PL](cudaStream_t st) { return layernorm_rows_launch(xx.p, oo.p, L.g, L.b, rows, xx.C, 1e-5f, st, PL); },
                   1, 0.0, 4.0 * rows * x.C * PL, "layernorm"});
  };
  // multi-head attention on the tensor cores: heads become "virtual images" of head-major, zero-padded copies of q, k
  // and V^T (head_dim -> multiple of 64, tokens -> multiple of 128); S = Q K^T and O = P V are batched GEMMs on the
  // tcgen05 kernel with a (masked) fp32 row softmax between them.  valid_k < 0: read m->ctx_len at launch time.
  auto mh_attention = [&](const Tensor& qsrc, int qcol, const Tensor& ksrc, int kcol, int vcol, int Tq, int Tk, int valid_k,
                          int heads, int d, Tensor* out, int Hh, int Ww, int Cc, int causal = 0) {
    if (rc) return;
    if (PL == 3) {
      // fp32-accurate mode: tiled fp32 attention straight on the q / k / v channel windows of the split-f16 tensors
      // (causal: the CLIP text encoder's self-attention, key tiles above the diagonal skipped)
      *out = talloc(B, Hh, Ww, Cc);
      flops += 4.0 * B * heads * (double)Tq * Tk * d;
      if (!dry) {
        const Tensor q_ = qsrc, k_ = ksrc, o_ = *out;
        ops.push_back({[m, q_, k_, o_, B, qcol, kcol, vcol, Tq, Tk, valid_k, heads, d, Cc, causal](cudaStream_t st) {
                         return attention_split_tiled_launch(q_.p, q_.C, qcol, k_.p, k_.C, kcol, vcol, o_.p, o_.C, Cc, B, Tq, Tk,
                                                             valid_k < 0 ? m->ctx_len : valid_k, heads, d, st, causal); },
                       2, 4.0 * B * heads * (double)Tq * Tk * d, 0.0,
                       causal ? "attention (fp32, tiled, causal, split-f16 operands)" : "attention (fp32, tiled, split-f16 operands)"});
      }
      return;
    }
    const int NV = B * heads;
    MhAttnShape sh;
    rc = mh_attention_shape(B, heads, Tq, Tk, d, &sh);
    if (rc) return;
    const int Tqp = sh.Tqp, Tkp = sh.Tkp, dpad = sh.dpad;
    Tensor qh = talloc(NV, 1, Tqp, dpad), kh = talloc(NV, 1, Tkp, dpad), vht = talloc(NV, 1, dpad, Tkp);
    Tensor oh = talloc(NV, 1, Tqp, dpad);
    *out = talloc(B, Hh, Ww, Cc);
    // fused attention unless B2E_FLASH=0 or head_dim > 192: the score matrix never leaves the SM (csrc/flash_attn.cu)
    static const bool flash_on = !(getenv("B2E_FLASH") && atoi(getenv("B2E_FLASH")) == 0);
    const bool fused = flash_on && dpad <= 192;
    rc = mh_attention_check(sh, fused, causal, valid_k, valid_k < 0);
    if (rc) return;
    Tensor sc;
    if (!fused) sc = talloc(NV, 1, Tqp, Tkp);   // materialised scores
    if (!dry) {
      MhAttnArgs aa;
      aa.q = qsrc.p; aa.q_pitch = qsrc.C; aa.q_col = qcol;
      aa.kv = ksrc.p; aa.kv_pitch = ksrc.C; aa.k_col = kcol; aa.v_col = vcol;
      aa.out = out->p; aa.out_pitch = out->C;
      aa.B = B; aa.Tq = Tq; aa.Tk = Tk; aa.heads = heads; aa.d = d;
      aa.valid_k = valid_k; aa.valid_k_live = valid_k < 0 ? &m->ctx_len : nullptr; aa.causal = causal;
      aa.qh = qh.p; aa.kh = kh.p; aa.vht = vht.p; aa.oh = oh.p; aa.sc = fused ? nullptr : sc.p;
      std::vector<AttnOp> aops;
      rc = mh_attention_ops(aa, fused, flash_attn_default_warps(), &aops);
      for (const AttnOp& o : aops) { ops.push_back({o.fn, o.kind, o.flops, o.bytes, o.desc}); flops += o.flops; }
    } else {
      flops += 4.0 * NV * (double)Tqp * Tkp * dpad;
    }
    tfree(qh); tfree(kh); tfree(vht);
    if (!fused) tfree(sc);
    tfree(oh);
  };
  if (m->clip) {
    // ---- CLIP text encoder: ids (B, L <= 128) -> (B, 1, 128, D) f16 token rows (rows >= L zero, masked as keys)
    const b2e_clip_config& cc = m->ccfg;
    const int D = cc.hidden_size, heads = cc.num_heads, d = D / heads;
    tfree(xin);
    Tensor x = talloc(B, 1, kCtxPad, D);
    if (!dry) {
      const Tensor xx = x;
      ops.push_back({[m, xx, B, D, PL](cudaStream_t st) {
                       return clip_embed_launch(m->in_ids, m->tok_emb, m->pos_emb, xx.p, B, m->ctx_len, kCtxPad, D, m->ccfg.vocab_size, st,
                                                PL); },
                     3, 0.0, (4.0 + 2.0 * PL) * B * kCtxPad * D, "token + position embedding"});
    }
    for (size_t li = 0; li < m->clayers.size() && !rc; ++li) {
      const b2e_unet::ClipL& L = m->clayers[li];
      Tensor a, qkv, o, x1, b2, f1, x2;
      lnorm(L.ln1, x, &a);
      conv(L.qkv, a, nullptr, 1, ConvEpilogue{}, &qkv, nullptr, nullptr, nullptr, false);
      tfree(a);
      mh_attention(qkv, 0, qkv, D, 2 * D, kCtxPad, kCtxPad, -1, heads, d, &o, 1, kCtxPad, D, 1);
      tfree(qkv);
      conv(L.out, o, nullptr, 1, ConvEpilogue{}, &x1, nullptr, &x, nullptr, false);
      tfree(o); tfree(x);
      lnorm(L.ln2, x1, &b2);
      conv(L.fc1, b2, nullptr, 1, ConvEpilogue{}, &f1, nullptr, nullptr, nullptr, false);
      tfree(b2);
      if (!dry && !rc) {
        const Tensor ff = f1;
        ops.push_back({[ff, PL](cudaStream_t st) { return quick_gelu_launch(ff.p, ff.p, (int64_t)(ff.bytes / sizeof(f16)), st, PL, ff.C); },
                       3, 0.0, 2.0 * (double)ff.bytes, "quick_gelu"});
      }
      conv(L.fc2, f1, nullptr, 1, ConvEpilogue{}, &x2, nullptr, &x1, nullptr, false);
      tfree(f1); tfree(x1);
      x = x2;
    }
    Tensor y;
    lnorm(m->clip_final_ln, x, &y);
    if (!dry && !rc) {
      const Tensor yy = y;
      ops.push_back({[m, yy, B, D, PL](cudaStream_t st) { return unpad_rows_f32_launch(yy.p, m->out_eps, B, m->ctx_len, kCtxPad, D, st, PL); },
                     3, 0.0, (4.0 + 2.0 * PL) * B * kCtxPad * D, "final hidden states -> fp32"});
    }
    if (rc) return rc;
    return finish_forward_only(m, ops_fwd, ar.peak, ws_bytes, need, dry, flops, B);
  }
  Tensor h;
  conv(m->conv_in, xin, nullptr, 1, ConvEpilogue{}, &h, nullptr);
  tfree(xin);
  std::vector<Tensor> stack;
  bool have_cat = false;
  Tensor cat;
  // a tensor that is still on the skip stack must outlive its consumer (dry-run addresses are
  // fake but unique per live allocation, so the same liveness logic applies)
  auto on_stack = [&](const Tensor& t) { for (auto& s : stack) if (s.p == t.p) return true; return false; };

  // gradient mode: what the backward pass needs from every node
  struct Save { Tensor x, h1, qkv, sc; float* st1 = nullptr; float* st2 = nullptr; };
  std::vector<Save> saves(m->nodes.size());
  int node_i = -1;
  for (const Node& nd : m->nodes) {
    if (rc) break;
    ++node_i;
    Save& sv = saves[node_i];
    switch (nd.kind) {
      case N_PUSH: stack.push_back(h); break;
      case N_POPCAT: cat = stack.back(); stack.pop_back(); have_cat = true; break;
      case N_RESNET: {
        const ResnetL& r = m->resnets[nd.idx];
        const Tensor* x1 = have_cat ? &cat : nullptr;
        Tensor a1, h1, a2, out;
        gnorm(r.n1, h, x1, 1, &a1, &sv.st1);
        ConvEpilogue e1;
        if (r.temb_off >= 0) { e1.temb = proj + r.temb_off; e1.temb_stride = m->sumC; }
        conv(r.c1, a1, nullptr, 1, e1, &h1, nullptr);
        tfree(a1);
        gnorm(r.n2, h1, nullptr, 1, &a2, &sv.st2);
        sv.x = h; sv.h1 = h1;
        const bool a2_view = a2.alias;          // a fused-GroupNorm view of h1: h1 must outlive conv2
        if (!a2_view) tfree(h1);
        // out = conv2(a2) + shortcut(x) : the block input rides along as a 1x1 K segment of conv2
        conv(r.c2, a2, nullptr, 1, ConvEpilogue{}, &out, nullptr, &h, x1);
        if (a2_view) tfree(h1);
        tfree(a2);
        if (!on_stack(h)) tfree(h);
        if (have_cat) { tfree(cat); have_cat = false; }
        h = out;
        break;
      }
      case N_ATTN: {
        const AttnL& a = m->attns[nd.idx];
        Tensor an, qkv, o, out;
        gnorm(a.gn, h, nullptr, 0, &an, &sv.st1);
        conv(a.qkv, an, nullptr, 1, ConvEpilogue{}, &qkv, nullptr, nullptr, nullptr, false);
        sv.x = h; sv.qkv = qkv;
        tfree(an);
        o = talloc(B, h.H, h.W, a.P, a.C);
        const int heads = c.attention_head_dim > 0 ? a.C / c.attention_head_dim : 1;
        const int T = h.H * h.W, C = a.P;   // C: padded width of q / k / v (zero tail: no effect on Q K^T, zero rows of V^T)
        if (PL == 3) {
          // fp32-accurate mode: fp32 attention core on the CUDA cores over the split-f16 q | k | v planes
          if (!dry) {
            const int Cr = a.C, dh = a.C / heads;
            if (sizeof(float) * 16 * (size_t)(dh + T) <= 160 * 1024 && qkv.C == 3 * C) {
              ops.push_back({[qkv, o, B, T, C, Cr, heads](cudaStream_t st) { return attention_split_launch(qkv.p, o.p, B, T, Cr, C, heads, st); },
                             2, 4.0 * B * (double)T * T * Cr, 0.0, "attention (fp32, split-f16 operands)"});
            } else {   // long sequences (decoder mid block: 4096 tokens): online softmax over key tiles
              ops.push_back({[qkv, o, B, T, C, Cr, heads, dh](cudaStream_t st) {
                               return attention_split_tiled_launch(qkv.p, qkv.C, 0, qkv.p, qkv.C, C, 2 * C, o.p, C, Cr, B, T, T, T, heads, dh, st); },
                             2, 4.0 * B * (double)T * T * Cr, 0.0, "attention (fp32, tiled, split-f16 operands)"});
            }
          }
          flops += 4.0 * B * (double)T * T * a.C;
        } else if (heads == 1 && single_head_attention_fits(B, h.H, h.W)) {
          // tensor-core attention: S = Q K^T and O = P V are batched GEMMs on the tcgen05 kernel (the per-image
          // B operand is read straight from the qkv tensor / a transposed copy of V); softmax in fp32 between
          Tensor sc = talloc(B, h.H, h.W, T);
          Tensor vt = talloc(B, 1, C, T);   // V^T: [N][C][T]
          sv.sc = sc;                       // P after the in-place softmax
          if (!dry) {
            std::vector<AttnOp> aops;
            rc = single_head_attention_ops(qkv.p, sc.p, vt.p, o.p, B, h.H, h.W, C, a.C, &aops);
            for (const AttnOp& op : aops) { ops.push_back({op.fn, op.kind, op.flops, op.bytes, op.desc}); flops += op.flops; }
          } else {
            flops += 4.0 * B * (double)T * T * C;
          }
          tfree(sc);
          tfree(vt);
        } else if (heads > 1 && (a.C / heads) % 8 == 0 && a.C / heads <= 192 && (T == 64 || (T % 128 == 0 && T <= 1024) || T == 4096) &&
                   !(getenv("B2E_FLASH") && atoi(getenv("B2E_FLASH")) == 0)) {
          // multi-head attention (LDM: 14-28 heads of 32 channels): fused tcgen05 attention over head-major copies
          const int d = a.C / heads;
          tfree(o);
          Tensor o2;
          mh_attention(qkv, 0, qkv, a.P, 2 * a.P, T, T, T, heads, d, &o2, h.H, h.W, a.P);
          o2.Cr = a.C;
          o = o2;
        } else if (heads > 1 && (a.C / heads) % 8 == 0 && a.C / heads <= 64 && T % 128 == 0 && T <= 1024 &&
                   conv_geometry(B * heads, h.H, h.W, T).Nt == 1) {
          // multi-head tensor-core attention: heads become "virtual images" v = n*heads + h of head-major copies of
          // q, k (head_dim zero-padded to one 64-channel K chunk) and V^T; S = Q K^T and O = P V are batched GEMMs on
          // the tcgen05 kernel, softmax in fp32 between them, heads merged back afterwards
          const int d = a.C / heads, NV = B * heads;
          Tensor qh = talloc(NV, h.H, h.W, 64), kh = talloc(NV, h.H, h.W, 64), vht = talloc(NV, 1, 64, T);
          Tensor sc = talloc(NV, h.H, h.W, T), oh = talloc(NV, h.H, h.W, 64);
          if (!dry) {
            ConvDesc d1;
            d1.s0.ptr = qh.p; d1.s0.C = 64;
            d1.N = NV; d1.H = h.H; d1.W = h.W; d1.ksize = 1; d1.stride = 1;
            d1.w_packed = kh.p; d1.b_batch_rows = T; d1.b_pitch = 64;      // K rows of virtual image v
            d1.Cout = T; d1.out_f16 = sc.p;
            ConvPlan p1;
            rc = conv_plan_build(&p1, d1);
            ConvDesc d2;
            d2.s0.ptr = sc.p; d2.s0.C = T;                                 // P
            d2.N = NV; d2.H = h.H; d2.W = h.W; d2.ksize = 1; d2.stride = 1;
            d2.w_packed = vht.p; d2.b_batch_rows = 64; d2.b_pitch = T;     // V^T rows of virtual image v
            d2.Cout = 64; d2.out_f16 = oh.p;
            ConvPlan p2;
            if (!rc) rc = conv_plan_build(&p2, d2);
            if (!rc) {
              const float scale = 1.0f / sqrtf((float)d);
              const int64_t rows = (int64_t)NV * T;
              const int P = a.P;
              ops.push_back({[qkv, qh, kh, vht, B, T, P, heads, d](cudaStream_t st) {
                               return split_heads_launch(qkv.p, qh.p, kh.p, vht.p, B, T, P, heads, d, st);
                             }, 3, 0.0, 2.0 * B * T * (3.0 * P + 3.0 * heads * 64)});
              ops.push_back({[p1](cudaStream_t st) { return conv_launch(p1, ConvEpilogue{}, st); }, 0, p1.flops, 0.0, "attention QK^T (heads batched)"});
              ops.push_back({[sc, rows, T, scale](cudaStream_t st) { return softmax_rows_launch(sc.p, rows, T, scale, st); },
                             3, 0.0, 4.0 * rows * T});
              ops.push_back({[p2](cudaStream_t st) { return conv_launch(p2, ConvEpilogue{}, st); }, 0, p2.flops, 0.0, "attention PV (heads batched)"});
              ops.push_back({[oh, o, B, T, P, heads, d](cudaStream_t st) { return merge_heads_launch(oh.p, o.p, B, T, P, heads, d, st); },
                             3, 0.0, 2.0 * B * T * (P + heads * 64.0)});
              flops += p1.flops + p2.flops;
            }
          } else {
            flops += 4.0 * NV * (double)T * T * 64;
          }
          tfree(qh); tfree(kh); tfree(vht); tfree(sc); tfree(oh);
        } else {
          if (!dry) {
            const int Cr = a.C;
            ops.push_back({[qkv, o, B, T, C, Cr, heads](cudaStream_t st) { return attention_launch(qkv.p, o.p, B, T, Cr, C, heads, st); },
                           2, 4.0 * B * (double)T * T * Cr, 0.0});
          }
          flops += 4.0 * B * (double)(h.H * h.W) * (h.H * h.W) * a.C;
        }
        tfree(qkv);
        conv(a.proj, o, nullptr, 1, ConvEpilogue{}, &out, nullptr, &h);
        tfree(o);
        if (!on_stack(h)) tfree(h);
        h = out;
        break;
      }
      case N_XFORMER: {
        const XfL& x = m->xfs[nd.idx];
        const int T = h.H * h.W, C = x.C;
        Tensor gn, t0, l1, qkv, o1, t1, l2, q2, kv, o2, t2, l3, f1, gg, t3, out;
        gnorm(x.gn, h, nullptr, 0, &gn, nullptr, 1e-6f);
        conv(x.proj_in, gn, nullptr, 1, ConvEpilogue{}, &t0, nullptr, nullptr, nullptr, false);
        tfree(gn);
        // self-attention
        lnorm(x.ln1, t0, &l1);
        conv(x.qkv1, l1, nullptr, 1, ConvEpilogue{}, &qkv, nullptr, nullptr, nullptr, false);
        tfree(l1);
        mh_attention(qkv, 0, qkv, C, 2 * C, T, T, T, x.heads, x.d, &o1, h.H, h.W, C);
        tfree(qkv);
        conv(x.out1, o1, nullptr, 1, ConvEpilogue{}, &t1, nullptr, &t0, nullptr, false);
        tfree(o1); tfree(t0);
        // cross-attention over the text tokens
        lnorm(x.ln2, t1, &l2);
        conv(x.q2, l2, nullptr, 1, ConvEpilogue{}, &q2, nullptr, nullptr, nullptr, false);
        tfree(l2);
        conv(x.kv2, ctxp, nullptr, 1, ConvEpilogue{}, &kv, nullptr, nullptr, nullptr, false);
        mh_attention(q2, 0, kv, 0, C, T, kCtxPad, -1, x.heads, x.d, &o2, h.H, h.W, C);
        tfree(q2); tfree(kv);
        conv(x.out2, o2, nullptr, 1, ConvEpilogue{}, &t2, nullptr, &t1, nullptr, false);
        tfree(o2); tfree(t1);
        // GEGLU feed-forward
        lnorm(x.ln3, t2, &l3);
        conv(x.ff1, l3, nullptr, 1, ConvEpilogue{}, &f1, nullptr, nullptr, nullptr, false);
        tfree(l3);
        gg = talloc(B, h.H, h.W, 4 * C);
        if (!dry) {
          const int64_t rows = (int64_t)B * T;
          ops.push_back({[f1, gg, rows, C, PL](cudaStream_t st) { return geglu_launch(f1.p, gg.p, rows, 4 * C, st, PL); }, 3, 0.0,
                         2.0 * rows * 12.0 * C, "geglu"});
        }
        tfree(f1);
        conv(x.ff2, gg, nullptr, 1, ConvEpilogue{}, &t3, nullptr, &t2, nullptr, false);
        tfree(gg); tfree(t2);
        conv(x.proj_out, t3, nullptr, 1, ConvEpilogue{}, &out, nullptr, &h);
        tfree(t3);
        if (!on_stack(h)) tfree(h);
        h = out;
        break;
      }
      case N_DOWN: {
        Tensor out;
        conv(m->downs[nd.idx], h, nullptr, 2, ConvEpilogue{}, &out, nullptr);
        if (!on_stack(h)) tfree(h);
        h = out;
        break;
      }
      case N_UP: {
        sv.x = h;
        if (up2_on && !keep && !h.alias && m->ups[nd.idx].w_up2 && h.H >= 64 && h.C == m->ups[nd.idx].cin_pad) {
          Tensor out;
          conv_up2(m->ups[nd.idx], h, &out);
          if (!on_stack(h)) tfree(h);
          h = out;
          break;
        }
        Tensor up = talloc(B, h.H * 2, h.W * 2, h.C, h.Cr), out;
        if (!dry) {
          Tensor hh = h;
          ops.push_back({[hh, up, B, PL](cudaStream_t st) { return upsample2x_launch(hh.p, up.p, B, hh.H, hh.W, hh.C * PL, st); },
                         3, 0.0, 10.0 * B * hh.H * hh.W * hh.C * PL});
        }
        if (!on_stack(h)) tfree(h);
        conv(m->ups[nd.idx], up, nullptr, 1, ConvEpilogue{}, &out, nullptr);
        tfree(up);
        h = out;
        break;
      }
    }
  }
  float* st_out = nullptr;
  Tensor h_last = h;
  if (!rc) {
    Tensor an;
    gnorm(m->norm_out, h, nullptr, 1, &an, &st_out);
    const bool an_view = an.alias;              // a fused-GroupNorm view of h: h must outlive conv_out
    if (!an_view) tfree(h);
    float dummy = 0.f;
    if (m->encoder) {
      // conv_out -> fp32 NCHW scratch -> quant_conv (1x1, fp32) -> the caller's output
      const int Q = m->enc_q, HWo = an.H * an.W;
      float* hq = (float*)ar.alloc(sizeof(float) * B * Q * HWo);
      ConvEpilogue eo;
      eo.out_f32_nchw = hq;
      conv(m->conv_out, an, nullptr, 1, eo, nullptr, nullptr);
      if (!dry && !rc)
        ops.push_back({[m, hq, B, Q, HWo](cudaStream_t st) { return pointwise_conv_f32_launch(hq, m->qc_w, m->qc_b, m->out_eps, B, Q, Q, HWo, st); },
                       3, 0.0, 8.0 * B * Q * HWo, "quant_conv 1x1 (fp32)"});
    } else {
      conv(m->conv_out, an, nullptr, 1, ConvEpilogue{}, nullptr, &dummy);
    }
    if (an_view) tfree(h);
    tfree(an);
  }
  // ---- backward program (decoder, gradient mode): d(loss)/d(latent) from d(loss)/d(image), walking the nodes in
  // reverse over the saved activations.  Every convolution gradient is the SAME tcgen05 implicit-GEMM kernel on the
  // dgrad twin of its weights; GroupNorm(+SiLU), softmax, upsample and the VQ front have their own backward kernels.
  if (!rc && m->grad) {
    if (!m->decoder) { set_error("unet: gradient mode is implemented for the VQ decoder only"); return B2E_UNSUPPORTED_SHAPE; }
    cur = &ops_bwd;
    const int So = S << (c.n_blocks - 1);
    float* gpart = (float*)ar.alloc(sizeof(float) * B * 64 * G * 2);
    auto gn_bwd = [&](const NormL& L, const Tensor& x, const float* stats, const Tensor& da, int silu, const Tensor* add,
                      Tensor* dx) {
      if (rc) return;
      *dx = talloc(B, x.H, x.W, x.C, x.Cr);
      if (dry) return;
      GNBwdArgs a;
      a.x = x.p; a.da = da.p; a.add = add ? add->p : nullptr; a.dx = dx->p;
      a.C = x.Cr; a.P = x.C; a.Pda = da.C; a.N = B; a.HW = x.H * x.W; a.G = G;
      a.gamma = L.g; a.beta = L.b; a.stats = stats; a.partial = gpart; a.chunks = gn_chunks(a.HW, a.C); a.silu = silu;
      if (add && add->C != x.C) { rc = B2E_INVALID_ARG; set_error("unet backward: residual pitch mismatch"); return; }
      ops.push_back({[a](cudaStream_t st) { return gn_bwd_launch(a, st); }, 1, 0.0, 10.0 * B * a.HW * a.C, "groupnorm backward"});
    };
    // gradient w.r.t. the image arrives as fp32 NCHW: pack to f16 NHWC with 64 (zero-padded) channels
    Tensor gy = talloc(B, So, So, kConvBlockK, c.out_channels);
    float* gs = (float*)ar.alloc(sizeof(float) * 4);   // gradient scale record (grad_scale_launch): keeps f16 gradients in range
    if (!dry) {
      const int Co = c.out_channels;
      cudaMemset(gs, 0, sizeof(float) * 4);
      ops.push_back({[m, gs, B, Co, So](cudaStream_t st) { return grad_scale_launch(m->in_dy, (int64_t)B * Co * So * So, gs, 1.f, st); },
                     3, 0.0, 4.0 * B * Co * So * So, "max|d(image)| -> power-of-two gradient scale"});
      ops.push_back({[m, gy, gs, B, Co, So](cudaStream_t st) { return pack_input_launch(m->in_dy, gy.p, B, Co, So, So, kConvBlockK, false, st, 1, gs); },
                     3, 0.0, (double)B * So * So * (4.0 * Co + 2.0 * kConvBlockK), "pack d(image)"});
    }
    Tensor d_an, g;
    conv(m->dgrads[m->conv_out_dg], gy, nullptr, 1, ConvEpilogue{}, &d_an, nullptr, nullptr, nullptr, false);
    gn_bwd(m->norm_out, h_last, st_out, d_an, 1, nullptr, &g);
    for (int ni = (int)m->nodes.size() - 1; ni >= 0 && !rc; --ni) {
      const Node& nd = m->nodes[ni];
      const Save& sv = saves[ni];
      switch (nd.kind) {
        case N_RESNET: {
          const ResnetL& r = m->resnets[nd.idx];
          Tensor d_a2, d_h1, d_a1, d_sc, gin;
          conv(m->dgrads[r.c2.dg], g, nullptr, 1, ConvEpilogue{}, &d_a2, nullptr, nullptr, nullptr, false);
          gn_bwd(r.n2, sv.h1, sv.st2, d_a2, 1, nullptr, &d_h1);
          conv(m->dgrads[r.c1.dg], d_h1, nullptr, 1, ConvEpilogue{}, &d_a1, nullptr, nullptr, nullptr, false);
          const Tensor* add = &g;   // identity shortcut
          if (r.has_sc) {
            conv(m->dgrads[r.sc_dg], g, nullptr, 1, ConvEpilogue{}, &d_sc, nullptr, nullptr, nullptr, false);
            add = &d_sc;
          }
          gn_bwd(r.n1, sv.x, sv.st1, d_a1, 1, add, &gin);
          g = gin;
          break;
        }
        case N_ATTN: {
          const AttnL& a = m->attns[nd.idx];
          const int T = sv.x.H * sv.x.W, P = a.P, Hh = sv.x.H, Ww = sv.x.W;
          if (!sv.sc.p && !dry) { rc = B2E_UNSUPPORTED_SHAPE; set_error("unet backward: attention needs the tensor-core path"); break; }
          Tensor dO, dV, dP, dQ, dK, d_an2, gin;
          conv(m->dgrads[a.proj.dg], g, nullptr, 1, ConvEpilogue{}, &dO, nullptr, nullptr, nullptr, false);
          Tensor Pt = talloc(B, Hh, Ww, T), dSt = talloc(B, Hh, Ww, T);
          Tensor dOt = talloc(B, 1, P, T), Kt = talloc(B, 1, P, T), Qt = talloc(B, 1, P, T);
          dV = talloc(B, Hh, Ww, P, a.C); dP = talloc(B, Hh, Ww, T); dQ = talloc(B, Hh, Ww, P, a.C); dK = talloc(B, Hh, Ww, P, a.C);
          if (!dry) {
            auto gemm = [&](const Tensor& A, int K, const f16* Bop, int brows, int bpitch, int Cout, const Tensor& out,
                            const char* what) {
              // out[n][t][co] = sum_k A[n][t][k] * Bop[n*brows + co][k]
              ConvDesc d;
              d.s0.ptr = A.p; d.s0.C = K; if (A.C != K) d.s0.pitch = A.C;
              d.N = B; d.H = Hh; d.W = Ww; d.ksize = 1; d.stride = 1;
              d.w_packed = Bop; d.b_batch_rows = brows; d.b_pitch = bpitch; d.Cout = Cout; d.out_f16 = out.p;
              ConvPlan pl;
              if (!rc) rc = conv_plan_build(&pl, d);
              if (!rc) { ops.push_back({[pl](cudaStream_t st) { return conv_launch(pl, ConvEpilogue{}, st); }, 0, pl.flops, 0.0, what}); flops += pl.flops; }
            };
            const Tensor sc = sv.sc, qkv = sv.qkv;
            const float scale = 1.0f / sqrtf((float)a.C);
            const int64_t rows = (int64_t)B * T;
            // dV = P^T dO
            ops.push_back({[sc, Pt, B, T](cudaStream_t st) { return transpose_window_launch(sc.p, Pt.p, B, T, T, T, 0, st); }, 3, 0.0, 4.0 * B * T * T, "P^T"});
            ops.push_back({[dO, dOt, B, T, P](cudaStream_t st) { return transpose_window_launch(dO.p, dOt.p, B, T, P, P, 0, st); }, 3, 0.0, 4.0 * B * T * P, "dO^T"});
            gemm(Pt, T, dOt.p, P, T, P, dV, "attention backward dV = P^T dO");
            // dP = dO V^T ; dS = scale * P o (dP - rowsum(dP o P))  (in place)
            gemm(dO, P, qkv.p + 2 * P, T, 3 * P, T, dP, "attention backward dP = dO V^T");
            ops.push_back({[sc, dP, rows, T, scale](cudaStream_t st) { return softmax_bwd_rows_launch(sc.p, dP.p, rows, T, scale, st); },
                           3, 0.0, 6.0 * rows * T, "softmax backward"});
            // dQ = dS K ; dK = dS^T Q
            ops.push_back({[qkv, Kt, B, T, P](cudaStream_t st) { return transpose_window_launch(qkv.p, Kt.p, B, T, P, 3 * P, P, st); }, 3, 0.0, 4.0 * B * T * P, "K^T"});
            gemm(dP, T, Kt.p, P, T, P, dQ, "attention backward dQ = dS K");
            ops.push_back({[dP, dSt, B, T](cudaStream_t st) { return transpose_window_launch(dP.p, dSt.p, B, T, T, T, 0, st); }, 3, 0.0, 4.0 * B * T * T, "dS^T"});
            ops.push_back({[qkv, Qt, B, T, P](cudaStream_t st) { return transpose_window_launch(qkv.p, Qt.p, B, T, P, 3 * P, 0, st); }, 3, 0.0, 4.0 * B * T * P, "Q^T"});
            gemm(dSt, T, Qt.p, P, T, P, dK, "attention backward dK = dS^T Q");
          }
          // d(normed input) = Wq^T dQ + Wk^T dK + Wv^T dV: one 1x1 convolution drawing K from three tensors
          conv(m->dgrads[a.qkv_dg], dQ, &dK, 1, ConvEpilogue{}, &d_an2, nullptr, &dV, nullptr, false);
          gn_bwd(a.gn, sv.x, sv.st1, d_an2, 0, &g, &gin);
          g = gin;
          break;
        }
        case N_UP: {
          Tensor d_up, gin = talloc(B, sv.x.H, sv.x.W, sv.x.C, sv.x.Cr);
          conv(m->dgrads[m->ups[nd.idx].dg], g, nullptr, 1, ConvEpilogue{}, &d_up, nullptr, nullptr, nullptr, false);
          if (!dry) {
            ops.push_back({[d_up, gin, B](cudaStream_t st) { return downsum2x_launch(d_up.p, gin.p, B, gin.H, gin.W, gin.C, st); },
                           3, 0.0, 10.0 * B * gin.H * gin.W * gin.C, "upsample backward"});
          }
          g = gin;
          break;
        }
        default: break;
      }
    }
    if (!rc) {
      Tensor dcols;
      conv(m->dgrads[m->conv_in_dg], g, nullptr, 1, ConvEpilogue{}, &dcols, nullptr, nullptr, nullptr, false);
      if (!dry && !rc) {
        const int L = c.in_channels;
        ops.push_back({[m, dcols, gs, B, L, S](cudaStream_t st) { return vq_col2im_bwd_launch(dcols.p, m->pq_w, m->out_dz, B, L, S, S, st, gs); },
                       3, 0.0, (double)B * S * S * (128.0 + 4.0 * L), "col2im + post_quant_conv backward (straight-through)"});
      }
    }
    cur = &ops_fwd;
  }
#undef ops
  if (rc) return rc;
  if (need) *need = ar.peak;
  if (!dry) {
    B2E_REQUIRE(ar.peak <= ws_bytes, B2E_WORKSPACE_TOO_SMALL, "unet: workspace too small (%zu > %zu)", ar.peak, ws_bytes);
    m->ops = std::move(ops_fwd);
    m->bops = std::move(ops_bwd);
    m->fwd_B = -1;
    m->flops = flops;
    m->cur_B = B;
  } else {
    m->flops = flops;
  }
  return B2E_OK;
}

// the common tail of every b2e_*_create: upload the weights, plan for max_batch (workspace size only), hand out the handle
int finish_create(b2e_unet* m, b2e_unet** out, const char* who) {
  int rc = build_model(m);
  if (!rc && cudaDeviceSynchronize() != cudaSuccess) { set_error("%s: device error", who); rc = B2E_CUDA_ERROR; }
  if (!rc) rc = build_program(m, (int)m->max_batch, nullptr, 0, &m->ws_need);
  if (rc) { delete m; return rc; }
  *out = m;
  return B2E_OK;
}

// the input-gradient op list of a classifier / face parser / LPIPS handle, over the live forward's activations
int run_backward(b2e_unet* m, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  for (auto& op : m->bops) {
    int rc = op.fn(st);
    if (rc) return rc;
  }
  return B2E_OK;
}

}  // namespace

extern "C" {

int b2e_unet_create(const b2e_unet_config* cfg, int64_t max_batch, b2e_unet** out) {
  B2E_REQUIRE(cfg && out && max_batch > 0, B2E_INVALID_ARG, "unet_create: bad argument");
  B2E_REQUIRE(cfg->n_blocks >= 1 && cfg->n_blocks <= 8, B2E_UNSUPPORTED_SHAPE, "unet_create: n_blocks");
  B2E_REQUIRE(cfg->in_channels <= 8 && cfg->out_channels <= 16, B2E_UNSUPPORTED_SHAPE,
              "unet_create: in_channels <= 8 and out_channels <= 16 required");
  for (int i = 0; i < cfg->n_blocks; ++i) {
    const int ch = cfg->block_out_channels[i];
    B2E_REQUIRE(ch % 8 == 0 && ch >= 32 && ch <= 2048 && ch % cfg->norm_num_groups == 0, B2E_UNSUPPORTED_SHAPE,
                "unet_create: block_out_channels must be multiples of 8 and of norm_num_groups, 32..2048 (got %d)", ch);
    B2E_REQUIRE(cfg->attention_head_dim <= 0 || !(cfg->down_attn[i] || cfg->up_attn[i]) || ch % cfg->attention_head_dim == 0,
                B2E_UNSUPPORTED_SHAPE, "unet_create: %d channels are not a multiple of attention_head_dim %d", ch,
                cfg->attention_head_dim);
  }
  B2E_REQUIRE(cfg->downsample_padding == 0 || cfg->downsample_padding == 1, B2E_UNSUPPORTED_SHAPE,
              "unet_create: downsample_padding must be 0 or 1");
  if (cfg->cross_attention_dim > 0) {
    B2E_REQUIRE(cfg->cross_attention_dim % 64 == 0 && cfg->num_attention_heads >= 1, B2E_UNSUPPORTED_SHAPE,
                "unet_create: cross_attention_dim must be a multiple of 64 and num_attention_heads >= 1");
    for (int i = 0; i < cfg->n_blocks; ++i) {
      const int ch = cfg->block_out_channels[i];
      B2E_REQUIRE(ch % 64 == 0 && ch % cfg->num_attention_heads == 0 && (ch / cfg->num_attention_heads) % 8 == 0,
                  B2E_UNSUPPORTED_SHAPE, "unet_create: conditional UNet needs channels %% 64 == 0 and head_dim %% 8 == 0 (got %d / %d heads)",
                  ch, cfg->num_attention_heads);
    }
  }
  B2E_REQUIRE(cfg->sample_size % (1 << (cfg->n_blocks - 1)) == 0, B2E_UNSUPPORTED_SHAPE, "unet_create: sample_size");
  B2E_REQUIRE(cfg->precision == 0 || cfg->precision == 1, B2E_INVALID_ARG, "unet_create: precision must be 0 (f16) or 1 (fp32-accurate)");
  if (cfg->precision == 1) {
    B2E_REQUIRE(cfg->in_channels == 1 || cfg->in_channels == 3 || cfg->in_channels == 4, B2E_UNSUPPORTED_SHAPE,
                "unet_create: the fp32-accurate mode needs 1, 3 or 4 input channels");
  }
  b2e_unet* m = new b2e_unet();
  m->cfg = *cfg;
  m->PL = cfg->precision == 1 ? 3 : 1;
  m->max_batch = max_batch;
  return finish_create(m, out, "unet_create");
}

int b2e_vqdec_create(const b2e_vqdec_config* cfg, int64_t max_batch, b2e_unet** out) {
  B2E_REQUIRE(cfg && out && max_batch > 0, B2E_INVALID_ARG, "vqdec_create: bad argument");
  B2E_REQUIRE(cfg->n_blocks >= 1 && cfg->n_blocks <= 8, B2E_UNSUPPORTED_SHAPE, "vqdec_create: n_blocks");
  B2E_REQUIRE((cfg->latent_channels == 1 || cfg->latent_channels == 3 || cfg->latent_channels == 4) && cfg->out_channels <= 16,
              B2E_UNSUPPORTED_SHAPE, "vqdec_create: latent_channels must be 1, 3 or 4 and out_channels <= 16");
  B2E_REQUIRE(cfg->num_vq_embeddings >= 0, B2E_INVALID_ARG, "vqdec_create: num_vq_embeddings");
  for (int i = 0; i < cfg->n_blocks; ++i) {
    const int ch = cfg->block_out_channels[i];
    B2E_REQUIRE(ch % 8 == 0 && ch >= 32 && ch <= 1024 && ch % cfg->norm_num_groups == 0, B2E_UNSUPPORTED_SHAPE,
                "vqdec_create: block_out_channels must be multiples of 8 and of norm_num_groups, 32..1024 (got %d)", ch);
  }
  B2E_REQUIRE(cfg->precision == 0 || cfg->precision == 1, B2E_INVALID_ARG, "vqdec_create: precision must be 0 (f16) or 1 (fp32-accurate)");
  b2e_unet* m = new b2e_unet();
  m->decoder = true;
  m->PL = cfg->precision == 1 ? 3 : 1;
  m->n_codes = cfg->num_vq_embeddings;
  b2e_unet_config& u = m->cfg;
  u = b2e_unet_config{};
  u.sample_size = cfg->sample_size; u.in_channels = cfg->latent_channels; u.out_channels = cfg->out_channels;
  u.n_blocks = cfg->n_blocks;
  for (int i = 0; i < cfg->n_blocks; ++i) u.block_out_channels[i] = cfg->block_out_channels[i];
  u.layers_per_block = cfg->layers_per_block; u.norm_num_groups = cfg->norm_num_groups; u.norm_eps = cfg->norm_eps;
  u.attention_head_dim = 0;
  m->max_batch = max_batch;
  return finish_create(m, out, "vqdec_create");
}

int b2e_vqenc_create(const b2e_vqenc_config* cfg, int64_t max_batch, b2e_unet** out) {
  B2E_REQUIRE(cfg && out && max_batch > 0, B2E_INVALID_ARG, "vqenc_create: bad argument");
  B2E_REQUIRE(cfg->n_blocks >= 1 && cfg->n_blocks <= 8, B2E_UNSUPPORTED_SHAPE, "vqenc_create: n_blocks");
  B2E_REQUIRE((cfg->in_channels == 1 || cfg->in_channels == 3 || cfg->in_channels == 4) && cfg->latent_channels >= 1 &&
                  cfg->latent_channels * (cfg->double_z ? 2 : 1) <= 16,
              B2E_UNSUPPORTED_SHAPE, "vqenc_create: in_channels must be 1, 3 or 4 and at most 16 output channels");
  B2E_REQUIRE(cfg->sample_size % (1 << (cfg->n_blocks - 1)) == 0, B2E_UNSUPPORTED_SHAPE, "vqenc_create: sample_size");
  for (int i = 0; i < cfg->n_blocks; ++i) {
    const int ch = cfg->block_out_channels[i];
    B2E_REQUIRE(ch % 8 == 0 && ch >= 32 && ch <= 1024 && ch % cfg->norm_num_groups == 0, B2E_UNSUPPORTED_SHAPE,
                "vqenc_create: block_out_channels must be multiples of 8 and of norm_num_groups, 32..1024 (got %d)", ch);
  }
  B2E_REQUIRE(cfg->precision == 0 || cfg->precision == 1, B2E_INVALID_ARG, "vqenc_create: precision must be 0 (f16) or 1 (fp32-accurate)");
  b2e_unet* m = new b2e_unet();
  m->encoder = true;
  m->PL = cfg->precision == 1 ? 3 : 1;
  m->enc_q = cfg->latent_channels * (cfg->double_z ? 2 : 1);
  b2e_unet_config& u = m->cfg;
  u = b2e_unet_config{};
  u.sample_size = cfg->sample_size; u.in_channels = cfg->in_channels; u.out_channels = m->enc_q;
  u.n_blocks = cfg->n_blocks;
  for (int i = 0; i < cfg->n_blocks; ++i) u.block_out_channels[i] = cfg->block_out_channels[i];
  u.layers_per_block = cfg->layers_per_block; u.norm_num_groups = cfg->norm_num_groups; u.norm_eps = cfg->norm_eps;
  u.attention_head_dim = 0; u.downsample_padding = 0;
  m->max_batch = max_batch;
  return finish_create(m, out, "vqenc_create");
}

int b2e_clip_create(const b2e_clip_config* cfg, int64_t max_batch, b2e_unet** out) {
  B2E_REQUIRE(cfg && out && max_batch > 0, B2E_INVALID_ARG, "clip_create: bad argument");
  B2E_REQUIRE(cfg->hidden_size % 64 == 0 && cfg->intermediate_size % 64 == 0 && cfg->num_heads >= 1 &&
                  cfg->hidden_size % cfg->num_heads == 0 && (cfg->hidden_size / cfg->num_heads) % 8 == 0 &&
                  cfg->hidden_size / cfg->num_heads <= 192 && cfg->hidden_size <= 2048,
              B2E_UNSUPPORTED_SHAPE, "clip_create: hidden / intermediate sizes must be multiples of 64, head_dim %% 8 == 0 and <= 192");
  B2E_REQUIRE(cfg->num_layers >= 1 && cfg->num_layers <= 64 && cfg->vocab_size >= 1 && cfg->max_positions >= 1 && cfg->max_positions <= 128,
              B2E_UNSUPPORTED_SHAPE, "clip_create: 1..64 layers, at most 128 positions");
  B2E_REQUIRE(cfg->precision == 0 || cfg->precision == 1, B2E_INVALID_ARG, "clip_create: precision must be 0 (f16) or 1 (fp32-accurate)");
  b2e_unet* m = new b2e_unet();
  m->clip = true;
  m->PL = cfg->precision == 1 ? 3 : 1;
  m->ccfg = *cfg;
  m->cfg = b2e_unet_config{};
  m->cfg.sample_size = 8; m->cfg.in_channels = 1; m->cfg.out_channels = 1; m->cfg.norm_num_groups = 1;
  m->max_batch = max_batch;
  return finish_create(m, out, "clip_create");
}

int b2e_clip_forward(b2e_unet* m, const int64_t* input_ids, int64_t seq_len, float* hidden, int64_t B, void* stream) {
  B2E_REQUIRE(m && input_ids && hidden, B2E_INVALID_ARG, "clip_forward: null pointer");
  B2E_REQUIRE(m->clip, B2E_INVALID_ARG, "clip_forward: not a text-encoder handle");
  B2E_REQUIRE(seq_len >= 1 && seq_len <= m->ccfg.max_positions, B2E_UNSUPPORTED_SHAPE, "clip_forward: %lld tokens (1..%d)",
              (long long)seq_len, m->ccfg.max_positions);
  m->in_ids = input_ids; m->ctx_len = (int)seq_len;
  return b2e_unet_forward(m, (const float*)input_ids, nullptr, hidden, B, stream);
}

int b2e_resnet_create(const b2e_resnet_config* cfg, int64_t max_batch, b2e_unet** out) {
  B2E_REQUIRE(cfg && out && max_batch > 0, B2E_INVALID_ARG, "resnet_create: bad argument");
  B2E_REQUIRE(cfg->in_channels >= 1 && cfg->in_channels <= 4, B2E_UNSUPPORTED_SHAPE, "resnet_create: 1..4 input channels");
  B2E_REQUIRE(cfg->input_size >= 64 && cfg->input_size % 64 == 0 && (cfg->input_size & (cfg->input_size - 1)) == 0,
              B2E_UNSUPPORTED_SHAPE, "resnet_create: input_size must be a power of two >= 64 (got %d)", cfg->input_size);
  B2E_REQUIRE(cfg->width >= 64 && cfg->width % 64 == 0 && cfg->num_classes >= 1 && cfg->num_classes <= 4096, B2E_UNSUPPORTED_SHAPE,
              "resnet_create: width must be a multiple of 64, 1..4096 classes");
  for (int i = 0; i < 4; ++i) B2E_REQUIRE(cfg->layers[i] >= 1 && cfg->layers[i] <= 64, B2E_UNSUPPORTED_SHAPE, "resnet_create: layers");
  b2e_unet* m = new b2e_unet();
  m->resnet = true;
  B2E_REQUIRE(cfg->head == 0 || (cfg->head == 1 && !cfg->bottleneck && cfg->width == 64 && cfg->num_classes <= 64),
              B2E_UNSUPPORTED_SHAPE, "resnet_create: the face-parser head needs a basic-block backbone of width 64 and <= 64 classes");
  m->grad = cfg->head == 0;   // the classifier exists for its input gradient (classifier guidance)
  B2E_REQUIRE(cfg->precision == 0 || cfg->precision == 1, B2E_INVALID_ARG, "resnet_create: precision must be 0 or 1");
  m->PL = cfg->precision == 1 ? 3 : 1;
  m->rcfg = *cfg;
  m->cfg = b2e_unet_config{};
  m->cfg.sample_size = cfg->input_size; m->cfg.in_channels = cfg->in_channels; m->cfg.out_channels = cfg->num_classes;
  m->max_batch = max_batch;
  return finish_create(m, out, "resnet_create");
}

int b2e_resnet_backward(b2e_unet* m, const float* d_logits, float* d_image, int64_t B, void* stream) {
  B2E_REQUIRE(m && d_logits && d_image, B2E_INVALID_ARG, "resnet_backward: null pointer");
  B2E_REQUIRE(m->resnet, B2E_INVALID_ARG, "resnet_backward: not a classifier / face-parser handle");
  B2E_REQUIRE(m->grad, B2E_INVALID_ARG, "resnet_backward: call b2e_unet_enable_grad first");
  B2E_REQUIRE(m->fwd_B == B && m->cur_B == B, B2E_INVALID_ARG,
              "resnet_backward: no live forward pass of batch %lld (last forward: %lld)", (long long)B, (long long)m->fwd_B);
  m->in_dlogits = d_logits; m->out_dz = d_image;
  return run_backward(m, stream);
}

static int unet_forward_impl(b2e_unet* m, const float* x, const int64_t* timesteps, float* eps, int64_t B, void* stream);

int b2e_resnet_forward_labels(b2e_unet* m, const float* x, int64_t* labels, int64_t B, void* stream) {
  B2E_REQUIRE(m && x && labels, B2E_INVALID_ARG, "resnet_forward_labels: null pointer");
  B2E_REQUIRE(m->resnet && m->rcfg.head == 1, B2E_INVALID_ARG, "resnet_forward_labels: not a face-parser handle");
  m->out_labels = labels;
  const int rc = unet_forward_impl(m, x, nullptr, reinterpret_cast<float*>(labels), B, stream);
  m->out_labels = nullptr;
  m->fwd_B = -1;     // no logits were produced: no backward over this pass
  return rc;
}

int b2e_lpips_create(const b2e_lpips_config* cfg, int64_t max_batch, b2e_unet** out) {
  B2E_REQUIRE(cfg && out && max_batch > 0, B2E_INVALID_ARG, "lpips_create: bad argument");
  B2E_REQUIRE(cfg->input_size >= 32 && cfg->input_size % 16 == 0 && cfg->input_size <= 4096, B2E_UNSUPPORTED_SHAPE,
              "lpips_create: input_size must be a multiple of 16 in 32..4096 (got %d)", cfg->input_size);
  B2E_REQUIRE(cfg->precision == 0 || cfg->precision == 1, B2E_INVALID_ARG, "lpips_create: precision must be 0 or 1");
  b2e_unet* m = new b2e_unet();
  m->lpips = true;
  m->grad = true;    // the regulariser exists for its input gradient
  m->PL = cfg->precision == 1 ? 3 : 1;
  m->lcfg = *cfg;
  m->cfg = b2e_unet_config{};
  m->cfg.sample_size = cfg->input_size; m->cfg.in_channels = 3; m->cfg.out_channels = 1;
  m->max_batch = max_batch;
  return finish_create(m, out, "lpips_create");
}

int b2e_lpips_set_reference(b2e_unet* m, const float* x_ref, int64_t B_ref, void* stream) {
  B2E_REQUIRE(m && x_ref, B2E_INVALID_ARG, "lpips_set_reference: null pointer");
  B2E_REQUIRE(m->lpips, B2E_INVALID_ARG, "lpips_set_reference: not an LPIPS handle");
  B2E_REQUIRE(m->ws, B2E_INVALID_ARG, "lpips_set_reference: no workspace bound");
  B2E_REQUIRE(B_ref >= 1 && B_ref <= m->max_batch, B2E_UNSUPPORTED_SHAPE, "lpips_set_reference: batch %lld (1..%lld)",
              (long long)B_ref, (long long)m->max_batch);
  if (B_ref != m->cur_B) {
    int rc = build_program(m, (int)B_ref, m->ws, m->ws_bytes, nullptr);
    if (rc) return rc;
  }
  m->in_x = x_ref; m->lp_mask = nullptr; m->lp_mask_batched = 0;
  m->lp_ref_mode = true;
  m->lp_ref_B = -1;
  m->fwd_B = -1;     // the activations now belong to the reference pass: no backward over them
  cudaStream_t st = (cudaStream_t)stream;
  int rc = B2E_OK;
  for (size_t i = 0; i < m->ops.size() && !rc; ++i) rc = m->ops[i].fn(st);
  m->lp_ref_mode = false;
  if (rc) return rc;
  m->lp_ref_B = B_ref;
  return B2E_OK;
}

int b2e_lpips_forward(b2e_unet* m, const float* x, const float* mask, int64_t mask_batch, float* dist, int64_t B, void* stream) {
  B2E_REQUIRE(m && x && dist, B2E_INVALID_ARG, "lpips_forward: null pointer");
  B2E_REQUIRE(m->lpips, B2E_INVALID_ARG, "lpips_forward: not an LPIPS handle");
  B2E_REQUIRE(!mask || mask_batch == 1 || mask_batch == B, B2E_UNSUPPORTED_SHAPE,
              "lpips_forward: the mask batch must be 1 or %lld (got %lld)", (long long)B, (long long)mask_batch);
  m->lp_mask = mask; m->lp_mask_batched = mask && mask_batch > 1;
  return unet_forward_impl(m, x, nullptr, dist, B, stream);
}

int b2e_lpips_backward(b2e_unet* m, const float* d_dist, float* d_x, int64_t B, void* stream) {
  B2E_REQUIRE(m && d_dist && d_x, B2E_INVALID_ARG, "lpips_backward: null pointer");
  B2E_REQUIRE(m->lpips, B2E_INVALID_ARG, "lpips_backward: not an LPIPS handle");
  B2E_REQUIRE(m->grad, B2E_INVALID_ARG, "lpips_backward: gradient mode is off (b2e_unet_enable_grad)");
  B2E_REQUIRE(m->fwd_B == B && m->cur_B == B, B2E_INVALID_ARG,
              "lpips_backward: no live forward pass of batch %lld (last forward: %lld)", (long long)B, (long long)m->fwd_B);
  m->in_dlogits = d_dist; m->out_dz = d_x;
  return run_backward(m, stream);
}

void b2e_unet_destroy(b2e_unet* m) { delete m; }

int b2e_unet_num_params(const b2e_unet* m) { return m ? (int)m->params.size() : 0; }

int b2e_unet_param_info(const b2e_unet* m, int idx, const char** name, int64_t* numel, int64_t* fan_in) {
  B2E_REQUIRE(m && idx >= 0 && idx < (int)m->params.size(), B2E_INVALID_ARG, "param_info: bad index");
  if (name) *name = m->params[idx].name.c_str();
  if (numel) *numel = m->params[idx].numel;
  if (fan_in) *fan_in = m->params[idx].fan_in;
  return B2E_OK;
}

int b2e_unet_set_param(b2e_unet* m, const char* name, const float* data, int64_t numel, void* stream) {
  B2E_REQUIRE(m && name && data, B2E_INVALID_ARG, "set_param: bad argument");
  auto it = m->pindex.find(name);
  B2E_REQUIRE(it != m->pindex.end(), B2E_NOT_FOUND, "set_param: unknown parameter '%s'", name);
  auto& p = m->params[it->second];
  B2E_REQUIRE(p.numel == numel, B2E_INVALID_ARG, "set_param: '%s' expects %lld elements, got %lld", name,
              (long long)p.numel, (long long)numel);
  return p.set(data, (cudaStream_t)stream);
}

size_t b2e_unet_workspace_bytes(const b2e_unet* m) { return m ? m->ws_need : 0; }

int b2e_unet_bind_workspace(b2e_unet* m, void* workspace, size_t workspace_bytes) {
  B2E_REQUIRE(m && workspace, B2E_INVALID_ARG, "bind_workspace: bad argument");
  B2E_REQUIRE(workspace_bytes >= m->ws_need, B2E_WORKSPACE_TOO_SMALL, "bind_workspace: need %zu bytes, got %zu",
              m->ws_need, workspace_bytes);
  B2E_REQUIRE(((uintptr_t)workspace & 255) == 0, B2E_INVALID_ARG, "bind_workspace: workspace must be 256-byte aligned");
  m->ws = workspace; m->ws_bytes = workspace_bytes;
  m->lp_ref_B = -1;
  return build_program(m, (int)m->max_batch, workspace, workspace_bytes, nullptr);
}

int b2e_unet_forward(b2e_unet* m, const float* x, const int64_t* timesteps, float* eps, int64_t B, void* stream) {
  // an LPIPS handle called directly (profiling): no input mask - the last b2e_lpips_forward's may be gone
  if (m && m->lpips) { m->lp_mask = nullptr; m->lp_mask_batched = 0; }
  return unet_forward_impl(m, x, timesteps, eps, B, stream);
}

static int unet_forward_impl(b2e_unet* m, const float* x, const int64_t* timesteps, float* eps, int64_t B, void* stream) {
  B2E_REQUIRE(m && x && (timesteps || m->decoder || m->encoder || m->resnet || m->clip || m->lpips) && eps, B2E_INVALID_ARG, "unet_forward: null pointer");
  B2E_REQUIRE(m->ws, B2E_INVALID_ARG, "unet_forward: no workspace bound");
  B2E_REQUIRE(B > 0 && B <= m->max_batch, B2E_UNSUPPORTED_SHAPE, "unet_forward: batch %lld exceeds max_batch %lld",
              (long long)B, (long long)m->max_batch);
  if (B != m->cur_B) {
    int rc = build_program(m, (int)B, m->ws, m->ws_bytes, nullptr);
    if (rc) return rc;
  }
  B2E_REQUIRE(m->cfg.cross_attention_dim <= 0 || m->in_ctx, B2E_INVALID_ARG,
              "unet_forward: a conditional UNet needs b2e_unet_forward_cond");
  B2E_REQUIRE(!m->lpips || m->lp_ref_B == 1 || m->lp_ref_B == B, B2E_INVALID_ARG,
              "lpips_forward: %s", m->lp_ref_B < 0 ? "no reference (b2e_lpips_set_reference)" : "the reference batch must be 1 or B");
  m->in_x = x; m->in_t = timesteps; m->out_eps = eps;
  cudaStream_t st = (cudaStream_t)stream;
  for (auto& op : m->ops) {
    int rc = op.fn(st);
    if (rc) return rc;
  }
  m->fwd_B = B;
  return B2E_OK;
}

int b2e_unet_forward_cond(b2e_unet* m, const float* x, const int64_t* timesteps, const float* context, int64_t ctx_len,
                          float* eps, int64_t B, void* stream) {
  B2E_REQUIRE(m && context, B2E_INVALID_ARG, "unet_forward_cond: null pointer");
  B2E_REQUIRE(m->cfg.cross_attention_dim > 0, B2E_INVALID_ARG, "unet_forward_cond: the model has no cross-attention");
  B2E_REQUIRE(ctx_len >= 1 && ctx_len <= 128, B2E_UNSUPPORTED_SHAPE, "unet_forward_cond: %lld context tokens (1..128)",
              (long long)ctx_len);
  m->in_ctx = context; m->ctx_len = (int)ctx_len;
  return b2e_unet_forward(m, x, timesteps, eps, B, stream);
}

int b2e_unet_enable_grad(b2e_unet* m, int enable) {
  B2E_REQUIRE(m, B2E_INVALID_ARG, "unet_enable_grad: null handle");
  B2E_REQUIRE(!enable || m->decoder || m->resnet || m->lpips, B2E_UNSUPPORTED_SHAPE,
              "unet_enable_grad: gradient mode is implemented for the VQ / KL decoder, the classifier and LPIPS");
  B2E_REQUIRE(!enable || m->PL == 1 || m->resnet || m->lpips, B2E_UNSUPPORTED_SHAPE, "unet_enable_grad: the fp32-accurate mode is forward-only");
  if ((enable != 0) == m->grad) return B2E_OK;
  m->grad = enable != 0;
  m->cur_B = -1; m->fwd_B = -1; m->ws = nullptr; m->ws_bytes = 0;   // the workspace must be re-queried and re-bound
  m->lp_ref_B = -1;
  return build_program(m, (int)m->max_batch, nullptr, 0, &m->ws_need);
}

int b2e_vqdec_backward(b2e_unet* m, const float* d_image, float* d_latent, int64_t B, void* stream) {
  B2E_REQUIRE(m && d_image && d_latent, B2E_INVALID_ARG, "vqdec_backward: null pointer");
  B2E_REQUIRE(m->decoder && m->grad, B2E_INVALID_ARG, "vqdec_backward: call b2e_unet_enable_grad on a VQ decoder first");
  B2E_REQUIRE(m->fwd_B == B && m->cur_B == B, B2E_INVALID_ARG,
              "vqdec_backward: no live forward pass of batch %lld (last forward: %lld)", (long long)B, (long long)m->fwd_B);
  m->in_dy = d_image; m->out_dz = d_latent;
  cudaStream_t st = (cudaStream_t)stream;
  // B2E_PROFILE_BWD=1: CUDA-event time of every backward op to stderr (diagnostic; synchronises)
  static const bool prof = getenv("B2E_PROFILE_BWD") && atoi(getenv("B2E_PROFILE_BWD")) != 0;
  if (prof) {
    std::vector<cudaEvent_t> ev(m->bops.size() + 1);
    for (auto& e : ev) cudaEventCreate(&e);
    cudaEventRecord(ev[0], st);
    int rc = B2E_OK;
    for (size_t i = 0; i < m->bops.size() && !rc; ++i) { rc = m->bops[i].fn(st); cudaEventRecord(ev[i + 1], st); }
    cudaStreamSynchronize(st);
    for (size_t i = 0; i < m->bops.size(); ++i) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, ev[i], ev[i + 1]);
      fprintf(stderr, "BWD %3zu %8.1f us %7.0f TF/s %7.0f GB/s  %s\n", i, ms * 1e3, m->bops[i].flops / (ms * 1e9 + 1e-9),
              m->bops[i].bytes / (ms * 1e6 + 1e-9), m->bops[i].desc.c_str());
    }
    for (auto& e : ev) cudaEventDestroy(e);
    return rc;
  }
  for (auto& op : m->bops) {
    int rc = op.fn(st);
    if (rc) return rc;
  }
  return B2E_OK;
}

const char* b2e_unet_op_desc(const b2e_unet* m, int idx) {
  if (!m || idx < 0 || idx >= (int)m->ops.size()) return "";
  return m->ops[idx].desc.c_str();
}

int b2e_unet_profile(b2e_unet* m, const float* x, const int64_t* timesteps, float* eps, int64_t B, void* stream,
                     int max_ops, int* n_ops, float* ms, double* flops, double* bytes, int* kind) {
  B2E_REQUIRE(m && x && (timesteps || m->decoder || m->encoder || m->resnet || m->clip || m->lpips) && eps && n_ops && ms && flops && bytes && kind, B2E_INVALID_ARG,
              "unet_profile: null pointer");
  // one plain pass first (plan rebuild / lazy function attributes), then the instrumented pass
  int rc = b2e_unet_forward(m, x, timesteps, eps, B, stream);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int n = (int)m->ops.size();
  B2E_REQUIRE(n <= max_ops, B2E_INVALID_ARG, "unet_profile: %d ops, room for %d", n, max_ops);
  std::vector<cudaEvent_t> ev(n + 1);
  for (auto& e : ev) B2E_CUDA(cudaEventCreate(&e));
  B2E_CUDA(cudaEventRecord(ev[0], st));
  for (int i = 0; i < n && !rc; ++i) {
    rc = m->ops[i].fn(st);
    cudaEventRecord(ev[i + 1], st);
  }
  cudaStreamSynchronize(st);
  for (int i = 0; i < n; ++i) {
    cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]);
    flops[i] = m->ops[i].flops; bytes[i] = m->ops[i].bytes; kind[i] = m->ops[i].kind;
  }
  for (auto& e : ev) cudaEventDestroy(e);
  *n_ops = n;
  return rc;
}

double b2e_unet_flops(const b2e_unet* m, int64_t B) {
  if (!m) return 0;
  const double per = m->flops / (double)(m->cur_B > 0 ? m->cur_B : m->max_batch);
  return per * (double)B;
}

int b2e_unet_launches_per_forward(const b2e_unet* m) {
  if (!m) return 0;
  // GroupNorm and the embedding MLP are two launches per op
  int n = 0;
  for (auto& op : m->ops) n += (op.kind == 1 || (op.kind == 3 && op.bytes == 0.0)) ? 2 : 1;
  return n;
}

}  // extern "C"
