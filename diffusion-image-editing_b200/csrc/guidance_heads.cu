// Loss heads of the network-based guidance functions: the part of NetAttrFunc / ClassifierAttrFunc that is not a
// dense network (SURVEY.md section 8, rows a12 / a13, Appendix A).  Each head returns the loss value AND its analytic
// gradient with respect to the network's output, so the caller seeds the network's backward pass with it
// (grad_output) instead of running softmax / sum / index autograd nodes.
//
//   NetAttrFunc.loss        src/attr_functions.py:213-219
//       p = softmax_c(logits[0]) ; area_c = sum_hw p[c] / (256*256) ; L = sum_{c in S} area_c
//       dL/dlogits[c,hw] = p[c,hw] * (1[c in S] - sum_{k in S} p[k,hw]) / (256*256)
//   ClassifierAttrFunc.loss src/attr_functions.py:237-257
//       a = logits.view(-1,40,2)[0] ; L = a[i][j] (+ (a[r][p] + score[p])^2)
//       dL/dlogits = onehot(2i+j) (+ 2 (a[r][p] + score[p]) onehot(2r+p)), other batch rows 0
// The batched entry points (per_sample=True) evaluate the same head on every image of a batch: loss[b] = L_b and one
// gradient per image, scaled by grad_scale (= loss_scale) as the last rounding step.
#include <cstdint>

#include "common.cuh"

namespace b2e {

constexpr int kHeadThreads = 256;
constexpr int kSegMaxClasses = 32;
constexpr int kClassifierLogits = 80;   // 40 attributes x 2

// one thread per pixel; logits are [B][C][HW] (class-major per image), so every per-class access is coalesced.
// blockIdx.y = image: the blocks of one image (and so its partial sums) do not depend on how many images the batch has
__global__ void __launch_bounds__(kHeadThreads)
seg_area_head_kernel(const float* __restrict__ logits, float* __restrict__ dlogits, double* __restrict__ partial,
                     int C, int64_t HW, uint32_t class_mask, float inv_div, float grad_scale) {
  pdl_wait();
  __shared__ double s_red[kHeadThreads / 32];
  const int64_t img = (int64_t)blockIdx.y * C * HW;
  logits += img;
  if (dlogits) dlogits += img;
  double acc = 0.0;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < HW; p += (int64_t)gridDim.x * blockDim.x) {
    float v[kSegMaxClasses];
    float m = -INFINITY;
#pragma unroll
    for (int c = 0; c < kSegMaxClasses; ++c)
      if (c < C) { v[c] = __ldcs(logits + (int64_t)c * HW + p); m = fmaxf(m, v[c]); }
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < kSegMaxClasses; ++c)
      if (c < C) { v[c] = expf(__fsub_rn(v[c], m)); s = __fadd_rn(s, v[c]); }
    float q = 0.f;   // probability mass of the selected classes at this pixel
#pragma unroll
    for (int c = 0; c < kSegMaxClasses; ++c)
      if (c < C) { v[c] = __fdiv_rn(v[c], s); if ((class_mask >> c) & 1u) q = __fadd_rn(q, v[c]); }
    acc += (double)q;
    if (dlogits) {
#pragma unroll
      for (int c = 0; c < kSegMaxClasses; ++c)
        if (c < C) {
          const float ind = ((class_mask >> c) & 1u) ? 1.f : 0.f;
          // grad_scale last: the rounding of autograd seeding loss_scale into the head's backward (x 1 is exact)
          __stcs(dlogits + (int64_t)c * HW + p,
                 __fmul_rn(__fmul_rn(__fmul_rn(v[c], __fsub_rn(ind, q)), inv_div), grad_scale));
        }
    }
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < kHeadThreads / 32; ++w) t += s_red[w];
    partial[(int64_t)blockIdx.y * gridDim.x + blockIdx.x] = t;
  }
}

// fixed-order final sum of each image's per-block partials (deterministic); one thread per image
__global__ void seg_area_final_kernel(const double* __restrict__ partial, int B, int n, float inv_div,
                                      float* __restrict__ loss) {
  pdl_wait();
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < B) {
    double t = 0.0;
    for (int i = 0; i < n; ++i) t += partial[(int64_t)b * n + i];
    loss[b] = (float)(t * (double)inv_div);
  }
}

__global__ void classifier_head_kernel(const float* __restrict__ logits, int64_t n, int idx, int ridx, float rscore,
                                       float* __restrict__ loss, float* __restrict__ dlogits) {
  pdl_wait();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float reg_t = 0.f;
  if (ridx >= 0) reg_t = __fadd_rn(logits[ridx], rscore);
  if (i < n && dlogits) {
    float g = 0.f;
    if (i == idx) g = 1.f;
    if (ridx >= 0 && i == ridx) g = __fadd_rn(g, __fmul_rn(2.f, reg_t));
    dlogits[i] = g;
  }
  if (i == 0 && loss) {
    float v = logits[idx];
    if (ridx >= 0) v = __fadd_rn(v, __fmul_rn(reg_t, reg_t));
    *loss = v;
  }
}

// one row of 80 logits per image: image b's loss and gradient row are the batch-1 head on that row; the gradient
// is multiplied by grad_scale as its last rounding step
__global__ void classifier_head_batched_kernel(const float* __restrict__ logits, int B, int idx, int ridx, float rscore,
                                               float grad_scale, float* __restrict__ loss, float* __restrict__ dlogits) {
  pdl_wait();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * kClassifierLogits) return;
  const int64_t b = i / kClassifierLogits;
  const int k = (int)(i - b * kClassifierLogits);
  const float* row = logits + b * kClassifierLogits;
  float reg_t = 0.f;
  if (ridx >= 0) reg_t = __fadd_rn(row[ridx], rscore);
  if (dlogits) {
    float g = 0.f;
    if (k == idx) g = 1.f;
    if (ridx >= 0 && k == ridx) g = __fadd_rn(g, __fmul_rn(2.f, reg_t));
    dlogits[i] = __fmul_rn(g, grad_scale);
  }
  if (k == 0 && loss) {
    float v = row[idx];
    if (ridx >= 0) v = __fadd_rn(v, __fmul_rn(reg_t, reg_t));
    loss[b] = v;
  }
}

}  // namespace b2e

using namespace b2e;

extern "C" {

size_t b2e_seg_area_head_batched_workspace_bytes(int64_t B) {
  return B < 1 ? 0 : sizeof(double) * kNumSMs * 8 * (size_t)B;
}

size_t b2e_seg_area_head_workspace_bytes(void) { return b2e_seg_area_head_batched_workspace_bytes(1); }

int b2e_seg_area_head_batched_f32(const float* logits, int64_t B, int64_t C, int64_t HW, const int32_t* classes,
                                  int n_classes, float area_divisor, float grad_scale, float* loss, float* dlogits,
                                  void* workspace, size_t workspace_bytes, void* stream) {
  B2E_REQUIRE(logits && loss && classes, B2E_INVALID_ARG, "seg_area_head: null pointer");
  B2E_REQUIRE(B >= 1 && B <= 65535, B2E_UNSUPPORTED_SHAPE, "seg_area_head: batch %lld (1 .. 65535)", (long long)B);
  B2E_REQUIRE(C >= 1 && C <= kSegMaxClasses, B2E_UNSUPPORTED_SHAPE, "seg_area_head: %lld classes (max %d)", (long long)C,
              kSegMaxClasses);
  B2E_REQUIRE(HW >= 1 && n_classes >= 0 && area_divisor > 0.f, B2E_INVALID_ARG, "seg_area_head: bad sizes");
  B2E_REQUIRE(workspace && workspace_bytes >= b2e_seg_area_head_batched_workspace_bytes(B), B2E_WORKSPACE_TOO_SMALL,
              "seg_area_head: workspace too small");
  uint32_t mask = 0;
  for (int i = 0; i < n_classes; ++i) {
    // a class listed twice counts twice in the reference (fancy indexing); refuse instead of silently differing
    B2E_REQUIRE(classes[i] >= 0 && classes[i] < C, B2E_INVALID_ARG, "seg_area_head: class id %d out of range", classes[i]);
    B2E_REQUIRE(!((mask >> classes[i]) & 1u), B2E_UNSUPPORTED_SHAPE, "seg_area_head: class id %d listed twice", classes[i]);
    mask |= 1u << classes[i];
  }
  cudaStream_t st = (cudaStream_t)stream;
  // blocks per image: a function of HW alone, so an image's partial sums (and loss bits) do not depend on the batch
  int grid = (int)((HW + kHeadThreads - 1) / kHeadThreads);
  if (grid > kNumSMs * 8) grid = kNumSMs * 8;
  const float inv_div = 1.f / area_divisor;   // 65536 in the reference: exact
  launch_pdl(seg_area_head_kernel, dim3(grid, (unsigned)B), dim3(kHeadThreads), 0, st, logits, dlogits, (double*)workspace,
             (int)C, HW, mask, inv_div, grad_scale);
  int rc = check_launch("seg_area_head");
  if (rc) return rc;
  launch_pdl(seg_area_final_kernel, dim3((unsigned)((B + 31) / 32)), dim3(32), 0, st, (const double*)workspace, (int)B, grid,
             inv_div, loss);
  return check_launch("seg_area_final");
}

int b2e_seg_area_head_f32(const float* logits, int64_t C, int64_t HW, const int32_t* classes, int n_classes,
                          float area_divisor, float* loss, float* dlogits, void* workspace, size_t workspace_bytes,
                          void* stream) {
  return b2e_seg_area_head_batched_f32(logits, 1, C, HW, classes, n_classes, area_divisor, 1.f, loss, dlogits, workspace,
                                       workspace_bytes, stream);
}

int b2e_classifier_head_f32(const float* logits, int64_t n, int idx_for_class, int idx_of_interest, int reg_idx,
                            int reg_pred, float reg_score, float* loss, float* dlogits, void* stream) {
  B2E_REQUIRE(logits && (loss || dlogits), B2E_INVALID_ARG, "classifier_head: null pointer");
  B2E_REQUIRE(n >= 80 && n % 80 == 0, B2E_UNSUPPORTED_SHAPE, "classifier_head: expected B x 80 logits, got %lld", (long long)n);
  B2E_REQUIRE(idx_for_class >= 0 && idx_for_class < 40 && (idx_of_interest == 0 || idx_of_interest == 1), B2E_INVALID_ARG,
              "classifier_head: index out of range");
  B2E_REQUIRE(reg_idx < 40 && (reg_idx < 0 || reg_pred == 0 || reg_pred == 1), B2E_INVALID_ARG,
              "classifier_head: regulariser index out of range");
  const int idx = 2 * idx_for_class + idx_of_interest, ridx = reg_idx >= 0 ? 2 * reg_idx + reg_pred : -1;
  launch_pdl(classifier_head_kernel, dim3((unsigned)((n + 127) / 128)), dim3(128), 0, (cudaStream_t)stream, logits, n, idx,
             ridx, reg_score, loss, dlogits);
  return check_launch("classifier_head");
}

int b2e_classifier_head_batched_f32(const float* logits, int64_t B, int idx_for_class, int idx_of_interest, int reg_idx,
                                    int reg_pred, float reg_score, float grad_scale, float* loss, float* dlogits,
                                    void* stream) {
  B2E_REQUIRE(logits && (loss || dlogits), B2E_INVALID_ARG, "classifier_head: null pointer");
  B2E_REQUIRE(B >= 1 && B <= (int64_t)INT32_MAX / kClassifierLogits, B2E_UNSUPPORTED_SHAPE,
              "classifier_head: batch %lld out of range", (long long)B);
  B2E_REQUIRE(idx_for_class >= 0 && idx_for_class < 40 && (idx_of_interest == 0 || idx_of_interest == 1), B2E_INVALID_ARG,
              "classifier_head: index out of range");
  B2E_REQUIRE(reg_idx < 40 && (reg_idx < 0 || reg_pred == 0 || reg_pred == 1), B2E_INVALID_ARG,
              "classifier_head: regulariser index out of range");
  const int idx = 2 * idx_for_class + idx_of_interest, ridx = reg_idx >= 0 ? 2 * reg_idx + reg_pred : -1;
  const int64_t n = B * kClassifierLogits;
  launch_pdl(classifier_head_batched_kernel, dim3((unsigned)((n + 127) / 128)), dim3(128), 0, (cudaStream_t)stream, logits,
             (int)B, idx, ridx, reg_score, grad_scale, loss, dlogits);
  return check_launch("classifier_head_batched");
}

}  // extern "C"
