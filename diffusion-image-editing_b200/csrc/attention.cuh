// Launch sequences of the tensor-core attention paths, shared by the UNet graph builder (csrc/unet.cu) and the
// b2e_attention_f16 test hook (csrc/attention.cu): padding rules, shape checks, plan building and launch order live
// here once.  A builder returns the launches as AttnOp records; the graph stores them, the hook runs them in order.
#pragma once
#include <functional>
#include <string>
#include <vector>

#include "unet_kernels.cuh"

namespace b2e {

// kind: 0 conv (tcgen05 GEMM), 2 attention, 3 other (the UNet op kinds)
struct AttnOp { std::function<int(cudaStream_t)> fn; int kind; double flops; double bytes; std::string desc; };

// Multi-head attention over head-major copies ("virtual images" v = image * heads + head).  Tokens are padded to
// 128-row blocks (a count below 128 becomes one block), head_dim d to dpad, the next multiple of 64.  qh .. sc: element
// counts of the temporaries (MhAttnArgs).
struct MhAttnShape { int Tqp, Tkp, dpad; size_t qh, kh, vht, oh, sc; };
int mh_attention_shape(int B, int heads, int Tq, int Tk, int d, MhAttnShape* s);
// refuses what the chosen path cannot run: head_dim > 192 on the fused kernel, causal attention on the materialised
// path, masked keys in a row the materialised softmax cannot hold (valid_k_live: the key count is only known at launch)
int mh_attention_check(const MhAttnShape& s, bool fused, int causal, int valid_k, bool valid_k_live);

struct MhAttnArgs {
  const f16* q; int q_pitch, q_col;              // q rows [B][Tq], head h at channels q_col + h*d
  const f16* kv; int kv_pitch, k_col, v_col;     // k / v rows [B][Tk] of one tensor
  f16* out; int out_pitch;                       // out rows [B][Tq]; the tail [heads*d, out_pitch) is zeroed
  int B, Tq, Tk, heads, d;
  int valid_k;                                   // keys >= valid_k are masked ...
  const int* valid_k_live = nullptr;             // ... or, if set, *valid_k_live read at every launch
  int causal = 0;                                // query i sees keys <= i (fused path only)
  // temporaries: qh [NV][Tqp][dpad], kh [NV][Tkp][dpad], vht [NV][dpad][Tkp], oh [NV][Tqp][dpad];
  // sc [NV][Tqp][Tkp] (materialised scores, fused == false only)
  f16 *qh, *kh, *vht, *oh, *sc;
};
// fused: gather -> flash_attn_kernel (dpad <= 192; softmax_warps 4 or 8) -> scatter.  Otherwise the materialised
// path: gather -> S = Q K^T (batched GEMM, 16-bit scores) -> masked row softmax -> O = P V (batched GEMM) -> scatter.
int mh_attention_ops(const MhAttnArgs& a, bool fused, int softmax_warps, std::vector<AttnOp>* ops);

// Single-head tensor-core attention straight from a packed qkv tensor [B][H*W][3C] (q | k | v blocks of C channels,
// zero tails beyond the d real ones) into out [B][H*W][C]: S = Q K^T (batched GEMM, 16-bit scores), row softmax,
// V^T copy, O = P V.  Temporaries sc [B][T][T], vt [B][C][T].
bool single_head_attention_fits(int B, int H, int W);
int single_head_attention_ops(const f16* qkv, f16* sc, f16* vt, f16* out, int B, int H, int W, int C, int d,
                              std::vector<AttnOp>* ops);

}  // namespace b2e
