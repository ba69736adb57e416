// Launch sequences of the tensor-core attention paths (see attention.cuh) and the b2e_attention_f16 test hook.
#include <math.h>

#include "attention.cuh"

namespace b2e {

int mh_attention_shape(int B, int heads, int Tq, int Tk, int d, MhAttnShape* s) {
  s->Tqp = Tq < 128 ? 128 : Tq;
  s->Tkp = Tk < 128 ? 128 : Tk;
  s->dpad = (d + 63) / 64 * 64;
  B2E_REQUIRE(Tq >= 1 && Tk >= 1 && s->Tqp % 128 == 0 && s->Tkp % 128 == 0 && (s->Tkp <= 1024 || s->Tkp == 2048 || s->Tkp == 4096),
              B2E_UNSUPPORTED_SHAPE, "attention over %d x %d tokens is not supported", Tq, Tk);
  B2E_REQUIRE(B >= 1 && heads >= 1 && d >= 8 && d % 8 == 0, B2E_UNSUPPORTED_SHAPE, "attention: %d heads of head_dim %d", heads, d);
  const size_t NV = (size_t)B * heads;
  s->qh = s->oh = NV * s->Tqp * s->dpad;
  s->kh = s->vht = NV * s->Tkp * s->dpad;
  s->sc = NV * s->Tqp * s->Tkp;
  return B2E_OK;
}

int mh_attention_check(const MhAttnShape& s, bool fused, int causal, int valid_k, bool valid_k_live) {
  B2E_REQUIRE(!fused || s.dpad <= 192, B2E_UNSUPPORTED_SHAPE, "attention: the fused kernel takes head_dim <= 192, not %d", s.dpad);
  B2E_REQUIRE(fused || !causal, B2E_UNSUPPORTED_SHAPE, "attention: causal attention needs the fused attention kernel");
  // the masked row softmax of the materialised path holds a row of at most 1024 scores
  B2E_REQUIRE(fused || valid_k_live || valid_k >= s.Tkp || s.Tkp <= 1024, B2E_UNSUPPORTED_SHAPE,
              "attention: %d of %d keys cannot be masked on the materialised path", valid_k, s.Tkp);
  return B2E_OK;
}

int mh_attention_ops(const MhAttnArgs& a, bool fused, int softmax_warps, std::vector<AttnOp>* ops) {
  MhAttnShape s;
  int rc = mh_attention_shape(a.B, a.heads, a.Tq, a.Tk, a.d, &s);
  if (!rc) rc = mh_attention_check(s, fused, a.causal, a.valid_k, a.valid_k_live != nullptr);
  if (rc) return rc;
  const int B = a.B, Tq = a.Tq, Tk = a.Tk, Tqp = s.Tqp, Tkp = s.Tkp, heads = a.heads, d = a.d, dpad = s.dpad;
  const int NV = B * heads;
  const float scale = 1.0f / sqrtf((float)d);
  const int valid_k = a.valid_k;
  const int* live = a.valid_k_live;
  const f16 *q = a.q, *kv = a.kv;
  f16 *qh = a.qh, *kh = a.kh, *vht = a.vht, *oh = a.oh, *out = a.out;
  const int qp = a.q_pitch, qcol = a.q_col, kp = a.kv_pitch, kcol = a.k_col, vcol = a.v_col, op = a.out_pitch;
  auto gathers = [&]() {
    ops->push_back({[q, qh, B, Tq, Tqp, qp, qcol, heads, d, dpad](cudaStream_t st) {
                      return gather_heads_launch(q, qh, B, Tq, Tqp, qp, qcol, heads, d, dpad, false, st); }, 3, 0.0, 4.0 * NV * Tqp * dpad, "gather q heads"});
    ops->push_back({[kv, kh, B, Tk, Tkp, kp, kcol, heads, d, dpad](cudaStream_t st) {
                      return gather_heads_launch(kv, kh, B, Tk, Tkp, kp, kcol, heads, d, dpad, false, st); }, 3, 0.0, 4.0 * NV * Tkp * dpad, "gather k heads"});
    ops->push_back({[kv, vht, B, Tk, Tkp, kp, vcol, heads, d, dpad](cudaStream_t st) {
                      return gather_heads_launch(kv, vht, B, Tk, Tkp, kp, vcol, heads, d, dpad, true, st); }, 3, 0.0, 4.0 * NV * Tkp * dpad, "gather V^T heads"});
  };
  auto scatter = [&]() {
    ops->push_back({[oh, out, B, Tq, Tqp, op, heads, d, dpad](cudaStream_t st) {
                      return scatter_heads_launch(oh, out, B, Tq, Tqp, op, heads, d, dpad, st); }, 3, 0.0, 4.0 * B * Tq * heads * d, "merge heads"});
  };
  if (fused) {
    // the score matrix never leaves the SM (csrc/flash_attn.cu)
    FlashPlan fp;
    rc = flash_attn_plan_build(&fp, qh, kh, vht, oh, NV, Tqp, Tkp, dpad);
    if (rc) return rc;
    const int causal = a.causal;
    gathers();
    ops->push_back({[fp, valid_k, live, scale, softmax_warps, causal](cudaStream_t st) {
                      return flash_attn_launch(fp, live ? *live : valid_k, scale, softmax_warps, st, causal); },
                    2, fp.flops, 0.0, "flash attention (tcgen05, S in TMEM)"});
    scatter();
    return B2E_OK;
  }
  f16* sc = a.sc;
  ConvDesc d1;
  d1.s0.ptr = qh; d1.s0.C = dpad;
  d1.N = NV; d1.H = 1; d1.W = Tqp; d1.ksize = 1; d1.stride = 1;
  d1.w_packed = kh; d1.b_batch_rows = Tkp; d1.b_pitch = dpad; d1.Cout = Tkp; d1.out_f16 = sc;
  ConvPlan p1;
  rc = conv_plan_build(&p1, d1);
  if (rc) return rc;
  ConvDesc d2;
  d2.s0.ptr = sc; d2.s0.C = Tkp;
  d2.N = NV; d2.H = 1; d2.W = Tqp; d2.ksize = 1; d2.stride = 1;
  d2.w_packed = vht; d2.b_batch_rows = dpad; d2.b_pitch = Tkp; d2.Cout = dpad; d2.out_f16 = oh;
  ConvPlan p2;
  rc = conv_plan_build(&p2, d2);
  if (rc) return rc;
  const int64_t rows = (int64_t)NV * Tqp;
  gathers();
  ops->push_back({[p1](cudaStream_t st) { return conv_launch(p1, ConvEpilogue{}, st); }, 0, p1.flops, 0.0, "attention QK^T (heads batched)"});
  ops->push_back({[sc, rows, Tkp, valid_k, live, scale](cudaStream_t st) {
                    return softmax_rows_masked_launch(sc, rows, Tkp, live ? *live : valid_k, scale, st); },
                  3, 0.0, 4.0 * rows * Tkp, "softmax"});
  ops->push_back({[p2](cudaStream_t st) { return conv_launch(p2, ConvEpilogue{}, st); }, 0, p2.flops, 0.0, "attention PV (heads batched)"});
  scatter();
  return B2E_OK;
}

bool single_head_attention_fits(int B, int H, int W) {
  const int T = H * W;
  return T % 128 == 0 && (T <= 1024 || T == 2048 || T == 4096) && conv_geometry(B, H, W, T).Nt == 1;
}

int single_head_attention_ops(const f16* qkv, f16* sc, f16* vt, f16* out, int B, int H, int W, int C, int d,
                              std::vector<AttnOp>* ops) {
  B2E_REQUIRE(single_head_attention_fits(B, H, W), B2E_UNSUPPORTED_SHAPE,
              "single-head attention: %d x %d x %d tokens do not fit the GEMM tiling", B, H, W);
  const int T = H * W;
  ConvDesc d1;
  d1.s0.ptr = qkv; d1.s0.C = C; d1.s0.pitch = 3 * C;                  // Q = channel window [0,C) of qkv
  d1.N = B; d1.H = H; d1.W = W; d1.ksize = 1; d1.stride = 1;
  d1.w_packed = qkv + C; d1.b_batch_rows = T; d1.b_pitch = 3 * C;    // K rows of image n
  d1.Cout = T; d1.out_f16 = sc;
  ConvPlan p1;
  int rc = conv_plan_build(&p1, d1);
  if (rc) return rc;
  ConvDesc d2;
  d2.s0.ptr = sc; d2.s0.C = T;                                        // P
  d2.N = B; d2.H = H; d2.W = W; d2.ksize = 1; d2.stride = 1;
  d2.w_packed = vt; d2.b_batch_rows = C; d2.b_pitch = T;              // V^T rows of image n
  d2.Cout = C; d2.out_f16 = out;
  ConvPlan p2;
  rc = conv_plan_build(&p2, d2);
  if (rc) return rc;
  const float scale = 1.0f / sqrtf((float)d);
  const int64_t rows = (int64_t)B * T;
  ops->push_back({[p1](cudaStream_t st) { return conv_launch(p1, ConvEpilogue{}, st); }, 0, p1.flops, 0.0, ""});
  ops->push_back({[sc, rows, T, scale](cudaStream_t st) { return softmax_rows_launch(sc, rows, T, scale, st); }, 3, 0.0, 4.0 * rows * T, ""});
  ops->push_back({[qkv, vt, B, T, C](cudaStream_t st) { return transpose_v_launch(qkv, vt, B, T, C, st); }, 3, 0.0, 4.0 * B * T * C, ""});
  ops->push_back({[p2](cudaStream_t st) { return conv_launch(p2, ConvEpilogue{}, st); }, 0, p2.flops, 0.0, ""});
  return B2E_OK;
}

}  // namespace b2e

using namespace b2e;

// Test hook: one attention through the engine's own launch sequence of the named path (include/b200edit.h).
extern "C" int b2e_attention_f16(const void* q, int64_t q_pitch, int64_t q_col, const void* kv, int64_t kv_pitch, int64_t k_col,
                                 int64_t v_col, void* out, int64_t out_pitch, int64_t B, int64_t H, int64_t W, int64_t Tk,
                                 int64_t valid_k, int64_t heads, int64_t head_dim, int causal, int path, int softmax_warps,
                                 void* stream) {
  B2E_REQUIRE(q && kv && out, B2E_INVALID_ARG, "attention: null pointer");
  B2E_REQUIRE(path >= B2E_ATTN_FUSED && path <= B2E_ATTN_FP32_TILED_CAUSAL, B2E_INVALID_ARG, "attention: unknown path %d", path);
  // path 6 is the causal instantiation of path 5's kernel: without causal = 1 it names no path
  B2E_REQUIRE(path != B2E_ATTN_FP32_TILED_CAUSAL || causal, B2E_INVALID_ARG,
              "attention: path %d with causal = 0 is an unknown path (the non-causal fp32 tiled kernel is path %d)", path,
              (int)B2E_ATTN_FP32_TILED);
  constexpr int64_t kMax = 1 << 30;
  B2E_REQUIRE(B >= 1 && H >= 1 && W >= 1 && Tk >= 1 && heads >= 1 && head_dim >= 1 && B * H * W < kMax && B * Tk < kMax &&
              heads * head_dim < kMax, B2E_INVALID_ARG, "attention: empty or oversized shape");
  B2E_REQUIRE(valid_k >= 1 && valid_k <= Tk, B2E_INVALID_ARG, "attention: valid_k %lld outside 1..%lld", (long long)valid_k,
              (long long)Tk);
  const int64_t C = heads * head_dim, Tq = H * W;
  B2E_REQUIRE(q_col >= 0 && k_col >= 0 && v_col >= 0 && q_col + C <= q_pitch && k_col + C <= kv_pitch && v_col + C <= kv_pitch &&
              C <= out_pitch && q_pitch < kMax && kv_pitch < kMax && out_pitch < kMax, B2E_INVALID_ARG,
              "attention: channel windows of %lld channels do not fit the pitches", (long long)C);
  B2E_REQUIRE(!causal || path == B2E_ATTN_FUSED || path == B2E_ATTN_FP32_TILED_CAUSAL, B2E_UNSUPPORTED_SHAPE,
              "attention: causal attention needs the fused path or the causal fp32 tiled path");
  B2E_REQUIRE(softmax_warps == 4 || softmax_warps == 8, B2E_INVALID_ARG, "attention: %d softmax warps (4 or 8)", softmax_warps);
  // the single-head, CUDA-core and fp32 split kernels read q | k | v blocks of one packed tensor [B][T][3P] and have no
  // key mask (self-attention over all tokens)
  if (path == B2E_ATTN_SINGLE_HEAD || path == B2E_ATTN_CUDA_CORE || path == B2E_ATTN_FP32_SPLIT) {
    B2E_REQUIRE(q == kv && q_pitch == kv_pitch && q_pitch == 3 * out_pitch && q_col == 0 && k_col == out_pitch &&
                v_col == 2 * out_pitch, B2E_UNSUPPORTED_SHAPE, "attention: path %d needs one packed qkv tensor [B][T][3 * out_pitch]", path);
    B2E_REQUIRE(Tk == Tq && valid_k == Tk, B2E_UNSUPPORTED_SHAPE, "attention: path %d is self-attention without a key mask", path);
  }
  if (path == B2E_ATTN_SINGLE_HEAD)
    B2E_REQUIRE(heads == 1 && single_head_attention_fits((int)B, (int)H, (int)W), B2E_UNSUPPORTED_SHAPE,
                "attention: single-head path for %lld heads over %lld x %lld x %lld tokens", (long long)heads, (long long)B,
                (long long)H, (long long)W);
  cudaStream_t st = (cudaStream_t)stream;
  int rc = B2E_OK;
  if (path == B2E_ATTN_CUDA_CORE) {
    rc = attention_launch((const f16*)q, (f16*)out, (int)B, (int)Tq, (int)C, (int)out_pitch, (int)heads, st);
    cudaStreamSynchronize(st);
    return rc;
  }
  if (path == B2E_ATTN_FP32_SPLIT) {
    rc = attention_split_launch((const f16*)q, (f16*)out, (int)B, (int)Tq, (int)C, (int)out_pitch, (int)heads, st);
    cudaStreamSynchronize(st);
    return rc;
  }
  if (path == B2E_ATTN_FP32_TILED || path == B2E_ATTN_FP32_TILED_CAUSAL) {
    rc = attention_split_tiled_launch((const f16*)q, (int)q_pitch, (int)q_col, (const f16*)kv, (int)kv_pitch, (int)k_col, (int)v_col,
                                      (f16*)out, (int)out_pitch, (int)C, (int)B, (int)Tq, (int)Tk, (int)valid_k, (int)heads,
                                      (int)head_dim, st, path == B2E_ATTN_FP32_TILED_CAUSAL);
    cudaStreamSynchronize(st);
    return rc;
  }
  // tensor-core paths: plans need the temporaries' addresses, so shapes are checked first and the plans built after
  // the allocation; nothing is launched before every plan is built
  std::vector<AttnOp> ops;
  char* mem = nullptr;
  size_t bytes = 0;
  if (path == B2E_ATTN_SINGLE_HEAD) {
    const size_t sc_b = sizeof(f16) * (size_t)B * Tq * Tq, vt_b = sizeof(f16) * (size_t)B * out_pitch * Tq;
    bytes = sc_b + vt_b;
    B2E_CUDA(cudaMalloc(&mem, bytes));
    rc = single_head_attention_ops((const f16*)q, (f16*)mem, (f16*)(mem + sc_b), (f16*)out, (int)B, (int)H, (int)W, (int)out_pitch,
                                   (int)head_dim, &ops);
  } else {
    const bool fused = path == B2E_ATTN_FUSED;
    MhAttnShape s;
    rc = mh_attention_shape((int)B, (int)heads, (int)Tq, (int)Tk, (int)head_dim, &s);
    if (!rc) rc = mh_attention_check(s, fused, causal, (int)valid_k, false);
    if (rc) return rc;
    const size_t q_b = sizeof(f16) * s.qh, o_b = sizeof(f16) * s.oh, k_b = sizeof(f16) * s.kh, v_b = sizeof(f16) * s.vht;
    const size_t sc_b = fused ? 0 : sizeof(f16) * s.sc;
    bytes = q_b + o_b + k_b + v_b + sc_b;
    B2E_CUDA(cudaMalloc(&mem, bytes));
    MhAttnArgs a;
    a.q = (const f16*)q; a.q_pitch = (int)q_pitch; a.q_col = (int)q_col;
    a.kv = (const f16*)kv; a.kv_pitch = (int)kv_pitch; a.k_col = (int)k_col; a.v_col = (int)v_col;
    a.out = (f16*)out; a.out_pitch = (int)out_pitch;
    a.B = (int)B; a.Tq = (int)Tq; a.Tk = (int)Tk; a.heads = (int)heads; a.d = (int)head_dim;
    a.valid_k = (int)valid_k; a.causal = causal;
    a.qh = (f16*)mem; a.oh = (f16*)(mem + q_b); a.kh = (f16*)(mem + q_b + o_b); a.vht = (f16*)(mem + q_b + o_b + k_b);
    a.sc = fused ? nullptr : (f16*)(mem + q_b + o_b + k_b + v_b);
    rc = mh_attention_ops(a, fused, softmax_warps, &ops);
  }
  for (size_t i = 0; i < ops.size() && !rc; ++i) rc = ops[i].fn(st);
  cudaStreamSynchronize(st);
  cudaFree(mem);
  return rc;
}
