// Mask path (integer-exact): MaskCreator.create_mask = per-class equality -> optional 7x7
// hard-max dilation -> sum over classes -> antialiased bilinear resize -> threshold ->
// channel replicate  (src/mask_creator.py:22-55, src/Morphology.py:47-111), plus the
// general Morphology.forward operator.
//
// The resize reproduces ATen's CPU `_upsample_bilinear2d_aa` bit for bit: fp32 triangle
// weights normalised per output (with the float/double promotions of the C++ source),
// W pass then H pass with an fp32 intermediate, and the compiled loop's accumulation
// order: acc = x0*w0; the next 4*floor((L-1)/4) taps as round(x*w) + acc, the remaining
// (L-1) mod 4 taps as fused multiply-adds (see oracle/mask.py).
#include <math.h>

#include "common.cuh"

namespace b2e {

constexpr int kMaxClasses = 32;

struct ClassSet {
  int n;
  int ids[kMaxClasses];
  float mult[kMaxClasses];  // multiplicity of a repeated class id
};

// m(y,x) = sum_c mult_c * max_{window}(seg == c), zero padding; map blockIdx.z of a batch of (H,W) maps
__global__ void class_dilate_sum_kernel(const int64_t* __restrict__ seg, float* __restrict__ out,
                                        int H, int W, int r, ClassSet cs) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= W || y >= H) return;
  seg += (int64_t)blockIdx.z * H * W;
  out += (int64_t)blockIdx.z * H * W;
  unsigned bits = 0;
  for (int dy = -r; dy <= r; ++dy) {
    const int yy = y + dy;
    if (yy < 0 || yy >= H) continue;
    for (int dx = -r; dx <= r; ++dx) {
      const int xx = x + dx;
      if (xx < 0 || xx >= W) continue;
      const int64_t v = __ldg(seg + (int64_t)yy * W + xx);
#pragma unroll 4
      for (int c = 0; c < cs.n; ++c) bits |= (v == (int64_t)cs.ids[c]) ? (1u << c) : 0u;
    }
  }
  float s = 0.f;
  for (int c = 0; c < cs.n; ++c)
    if (bits & (1u << c)) s = __fadd_rn(s, cs.mult[c]);
  out[(int64_t)y * W + x] = s;
}

// ---- ATen HelperInterpLinear::_compute_indices_min_size_weights_aa, scalar_t = float
struct AATable {
  int* xmin;     // [out]
  int* xsize;    // [out]
  float* w;      // [out][max_taps]
  int max_taps;
};

__host__ __device__ inline int aa_max_taps(int64_t in_size, int64_t out_size) {
  float scale = (float)in_size / (float)out_size;
  float support = (scale >= 1.0f) ? (float)(1.0 * (double)scale) : 1.0f;
  return (int)ceilf(support) * 2 + 1;
}

__global__ void aa_weights_kernel(int in_size, int out_size, AATable t) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= out_size) return;
  const float scale = __fdiv_rn((float)in_size, (float)out_size);
  const float support = (scale >= 1.0f) ? scale : 1.0f;
  const float invscale = (scale >= 1.0f) ? (float)__ddiv_rn(1.0, (double)scale) : 1.0f;
  const float center = (float)__dmul_rn((double)scale, (double)i + 0.5);
  long long xmin = (long long)__dadd_rn((double)__fsub_rn(center, support), 0.5);
  if (xmin < 0) xmin = 0;
  long long xmax = (long long)__dadd_rn((double)__fadd_rn(center, support), 0.5);
  if (xmax > in_size) xmax = in_size;
  long long xsize = xmax - xmin;
  if (xsize < 0) xsize = 0;
  if (xsize > t.max_taps) xsize = t.max_taps;
  float* w = t.w + (size_t)i * t.max_taps;
  float total = 0.f;
  for (int j = 0; j < (int)xsize; ++j) {
    const float d = __fsub_rn((float)(j + xmin), center);
    float x = (float)__dmul_rn(__dadd_rn((double)d, 0.5), (double)invscale);
    x = fabsf(x);
    const float wj = (x < 1.0f) ? (float)__dsub_rn(1.0, (double)x) : 0.f;
    w[j] = wj;
    total = __fadd_rn(total, wj);
  }
  if (total != 0.f)
    for (int j = 0; j < (int)xsize; ++j) w[j] = __fdiv_rn(w[j], total);
  for (int j = (int)xsize; j < t.max_taps; ++j) w[j] = 0.f;
  t.xmin[i] = (int)xmin;
  t.xsize[i] = (int)xsize;
}

__device__ __forceinline__ float aa_accumulate(const float* __restrict__ src, int64_t stride,
                                               const float* __restrict__ w, int n) {
  float acc = __fmul_rn(src[0], w[0]);
  const int n_plain = 4 * ((n - 1) / 4);
  int j = 1;
  for (; j <= n_plain; ++j) acc = __fadd_rn(acc, __fmul_rn(src[(int64_t)j * stride], w[j]));
  for (; j < n; ++j) acc = __fmaf_rn(src[(int64_t)j * stride], w[j], acc);
  return acc;
}

// horizontal: in (H,W) -> tmp (H,ow); plane blockIdx.z of a batch
__global__ void aa_resize_h_kernel(const float* __restrict__ in, float* __restrict__ tmp, int H,
                                   int W, int ow, AATable t) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  if (i >= ow || y >= H) return;
  in += (int64_t)blockIdx.z * H * W;
  tmp += (int64_t)blockIdx.z * H * ow;
  const int n = t.xsize[i];
  tmp[(int64_t)y * ow + i] =
      n > 0 ? aa_accumulate(in + (int64_t)y * W + t.xmin[i], 1, t.w + (size_t)i * t.max_taps, n) : 0.f;
}

// vertical: tmp (H,ow) -> out; threshold != 0: out = (r >= 1) replicated over `channels`; plane blockIdx.z
__global__ void aa_resize_v_kernel(const float* __restrict__ tmp, float* __restrict__ out, int H,
                                   int ow, int oh, AATable t, int threshold, int channels) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= ow || i >= oh) return;
  tmp += (int64_t)blockIdx.z * H * ow;
  out += (int64_t)blockIdx.z * (threshold ? channels : 1) * oh * ow;
  const int n = t.xsize[i];
  float r = n > 0 ? aa_accumulate(tmp + (int64_t)t.xmin[i] * ow + x, ow, t.w + (size_t)i * t.max_taps, n)
                  : 0.f;
  if (threshold) {
    // mask[mask < 1] = 0 ; mask[mask > 1] = 1   (src/mask_creator.py:52-53)
    r = (r < 1.f) ? 0.f : ((r > 1.f) ? 1.f : r);
    for (int c = 0; c < channels; ++c) out[((int64_t)c * oh + i) * ow + x] = r;
  } else {
    out[(int64_t)i * ow + x] = r;
  }
}

// Morphology.forward: zero pad k/2, window max of (w + x) [dilation] or -(max (w - x)) [erosion];
// soft: logsumexp(beta*v)/beta                                  (src/Morphology.py:47-84)
__global__ void morphology_kernel(const float* __restrict__ x, const float* __restrict__ wgt,
                                  float* __restrict__ out, int B, int Cin, int Cout, int H, int W,
                                  int k, int op, int soft, float beta) {
  const int xo = blockIdx.x * blockDim.x + threadIdx.x;
  const int yo = blockIdx.y * blockDim.y + threadIdx.y;
  const int bc = blockIdx.z;
  if (xo >= W || yo >= H) return;
  const int b = bc / Cout, co = bc % Cout;
  const int p = (k - 1) / 2;  // fixed_padding: pad_beg = (k-1)//2
  float m = -INFINITY;
  // pass 1: max
  for (int ci = 0; ci < Cin; ++ci)
    for (int dy = 0; dy < k; ++dy)
      for (int dx = 0; dx < k; ++dx) {
        const int yy = yo + dy - p, xx = xo + dx - p;
        const float xv = (yy >= 0 && yy < H && xx >= 0 && xx < W)
                             ? __ldg(x + (((int64_t)b * Cin + ci) * H + yy) * W + xx) : 0.f;
        const float wv = __ldg(wgt + (((int64_t)co * Cin + ci) * k + dy) * k + dx);
        float v = op == 0 ? __fadd_rn(wv, xv) : __fsub_rn(wv, xv);
        if (soft) v = __fmul_rn(v, beta);
        m = fmaxf(m, v);
      }
  float r = m;
  if (soft) {
    float s = 0.f;
    for (int ci = 0; ci < Cin; ++ci)
      for (int dy = 0; dy < k; ++dy)
        for (int dx = 0; dx < k; ++dx) {
          const int yy = yo + dy - p, xx = xo + dx - p;
          const float xv = (yy >= 0 && yy < H && xx >= 0 && xx < W)
                               ? __ldg(x + (((int64_t)b * Cin + ci) * H + yy) * W + xx) : 0.f;
          const float wv = __ldg(wgt + (((int64_t)co * Cin + ci) * k + dy) * k + dx);
          float v = __fmul_rn(op == 0 ? __fadd_rn(wv, xv) : __fsub_rn(wv, xv), beta);
          s += expf(v - m);
        }
    r = (m + logf(s)) / beta;
  }
  if (op == 1) r = -r;
  out[(((int64_t)b * Cout + co) * H + yo) * W + xo] = r;
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// N maps: one (H,W) class-sum plane and one (H,ow) intermediate each; the weight tables depend only on the sizes
// and are shared.  N = 1 is the single-map layout.
struct MaskWs {
  float* plane;  // (N,H,W) class-sum
  float* tmp;    // (N,H,ow)
  AATable th, tv;
  size_t bytes;
};

static MaskWs carve(void* ws, int64_t N, int64_t H, int64_t W, int64_t oh, int64_t ow) {
  MaskWs m;
  char* p = (char*)ws;
  size_t off = 0;
  auto take = [&](size_t n) { char* q = p ? p + off : nullptr; off += align_up(n, 256); return q; };
  m.plane = (float*)take(sizeof(float) * N * H * W);
  m.tmp = (float*)take(sizeof(float) * N * H * ow);
  m.th.max_taps = aa_max_taps(W, ow);
  m.tv.max_taps = aa_max_taps(H, oh);
  m.th.xmin = (int*)take(sizeof(int) * ow);
  m.th.xsize = (int*)take(sizeof(int) * ow);
  m.th.w = (float*)take(sizeof(float) * ow * m.th.max_taps);
  m.tv.xmin = (int*)take(sizeof(int) * oh);
  m.tv.xsize = (int*)take(sizeof(int) * oh);
  m.tv.w = (float*)take(sizeof(float) * oh * m.tv.max_taps);
  m.bytes = off;
  return m;
}

static int run_resize(const float* in, int64_t N, int64_t H, int64_t W, float* out, int64_t oh, int64_t ow,
                      const MaskWs& m, int threshold, int channels, cudaStream_t st) {
  aa_weights_kernel<<<(unsigned)((ow + 127) / 128), 128, 0, st>>>((int)W, (int)ow, m.th);
  int rc = check_launch("aa_weights(h)");
  if (rc) return rc;
  aa_weights_kernel<<<(unsigned)((oh + 127) / 128), 128, 0, st>>>((int)H, (int)oh, m.tv);
  rc = check_launch("aa_weights(v)");
  if (rc) return rc;
  dim3 blk(32, 8);
  aa_resize_h_kernel<<<dim3((unsigned)((ow + 31) / 32), (unsigned)((H + 7) / 8), (unsigned)N), blk, 0, st>>>(
      in, m.tmp, (int)H, (int)W, (int)ow, m.th);
  rc = check_launch("aa_resize_h");
  if (rc) return rc;
  aa_resize_v_kernel<<<dim3((unsigned)((ow + 31) / 32), (unsigned)((oh + 7) / 8), (unsigned)N), blk, 0, st>>>(
      m.tmp, out, (int)H, (int)ow, (int)oh, m.tv, threshold, channels);
  return check_launch("aa_resize_v");
}

}  // namespace b2e

using namespace b2e;

extern "C" {

size_t b2e_mask_workspace_bytes(int64_t H, int64_t W, int64_t out_h, int64_t out_w) {
  if (H <= 0 || W <= 0 || out_h <= 0 || out_w <= 0) return 0;
  return carve(nullptr, 1, H, W, out_h, out_w).bytes;
}

size_t b2e_mask_batched_workspace_bytes(int64_t N, int64_t H, int64_t W, int64_t out_h, int64_t out_w) {
  if (N <= 0 || H <= 0 || W <= 0 || out_h <= 0 || out_w <= 0) return 0;
  return carve(nullptr, N, H, W, out_h, out_w).bytes;
}

int b2e_mask_from_seg(const int64_t* seg, int64_t H, int64_t W, const int32_t* classes,
                      int n_classes, int dilate, int ksize, int64_t out_h, int64_t out_w,
                      int channels, int antialias, float* out, void* workspace,
                      size_t workspace_bytes, void* stream) {
  return b2e_mask_from_seg_batched(seg, 1, H, W, classes, n_classes, dilate, ksize, out_h, out_w, channels, antialias, out,
                                   workspace, workspace_bytes, stream);
}

int b2e_mask_from_seg_batched(const int64_t* seg, int64_t N, int64_t H, int64_t W, const int32_t* classes,
                              int n_classes, int dilate, int ksize, int64_t out_h, int64_t out_w,
                              int channels, int antialias, float* out, void* workspace,
                              size_t workspace_bytes, void* stream) {
  B2E_REQUIRE(seg && out && workspace, B2E_INVALID_ARG, "mask_from_seg: null pointer");
  B2E_REQUIRE(N > 0 && N < 65536 && H > 0 && W > 0 && out_h > 0 && out_w > 0 && channels > 0, B2E_UNSUPPORTED_SHAPE,
              "mask_from_seg: bad shape");
  B2E_REQUIRE(H < (1 << 15) && W < (1 << 15), B2E_UNSUPPORTED_SHAPE, "mask_from_seg: map too large");
  B2E_REQUIRE(n_classes >= 0 && (n_classes == 0 || classes), B2E_INVALID_ARG, "mask_from_seg: classes");
  B2E_REQUIRE(!dilate || (ksize % 2 == 1 && ksize >= 1 && ksize <= 31), B2E_UNSUPPORTED_SHAPE,
              "mask_from_seg: dilation kernel size must be odd and <= 31 (got %d)", ksize);
  B2E_REQUIRE(antialias, B2E_UNSUPPORTED_SHAPE,
              "mask_from_seg: only the antialiased resize (torchvision >= 0.17 default) is implemented");
  B2E_REQUIRE(workspace_bytes >= b2e_mask_batched_workspace_bytes(N, H, W, out_h, out_w), B2E_WORKSPACE_TOO_SMALL,
              "mask_from_seg: workspace too small");
  ClassSet cs;
  cs.n = 0;
  for (int i = 0; i < n_classes; ++i) {
    int j = 0;
    for (; j < cs.n; ++j)
      if (cs.ids[j] == classes[i]) break;
    if (j == cs.n) {
      B2E_REQUIRE(cs.n < kMaxClasses, B2E_UNSUPPORTED_SHAPE, "mask_from_seg: more than %d distinct classes",
                  kMaxClasses);
      cs.ids[cs.n] = classes[i];
      cs.mult[cs.n] = 0.f;
      ++cs.n;
    }
    cs.mult[j] += 1.f;
  }
  cudaStream_t st = (cudaStream_t)stream;
  MaskWs m = carve(workspace, N, H, W, out_h, out_w);
  dim3 blk(32, 8);
  class_dilate_sum_kernel<<<dim3((unsigned)((W + 31) / 32), (unsigned)((H + 7) / 8), (unsigned)N), blk, 0, st>>>(
      seg, m.plane, (int)H, (int)W, dilate ? ksize / 2 : 0, cs);
  int rc = check_launch("class_dilate_sum");
  if (rc) return rc;
  return run_resize(m.plane, N, H, W, out, out_h, out_w, m, 1, channels, st);
}

int b2e_resize_bilinear_aa_f32(const float* in, int64_t H, int64_t W, float* out, int64_t out_h,
                               int64_t out_w, void* workspace, size_t workspace_bytes, void* stream) {
  B2E_REQUIRE(in && out && workspace, B2E_INVALID_ARG, "resize: null pointer");
  B2E_REQUIRE(H > 0 && W > 0 && out_h > 0 && out_w > 0, B2E_UNSUPPORTED_SHAPE, "resize: bad shape");
  B2E_REQUIRE(workspace_bytes >= b2e_mask_workspace_bytes(H, W, out_h, out_w), B2E_WORKSPACE_TOO_SMALL,
              "resize: workspace too small");
  MaskWs m = carve(workspace, 1, H, W, out_h, out_w);
  return run_resize(in, 1, H, W, out, out_h, out_w, m, 0, 1, (cudaStream_t)stream);
}

int b2e_morphology2d_f32(const float* x, const float* weight, float* out, int64_t B, int64_t Cin,
                         int64_t Cout, int64_t H, int64_t W, int ksize, int op, int soft,
                         float beta, void* stream) {
  B2E_REQUIRE(x && weight && out, B2E_INVALID_ARG, "morphology: null pointer");
  B2E_REQUIRE(B > 0 && Cin > 0 && Cout > 0 && H > 0 && W > 0 && ksize >= 1 && B * Cout < 65536,
              B2E_UNSUPPORTED_SHAPE, "morphology: bad shape");
  B2E_REQUIRE(op == 0 || op == 1, B2E_INVALID_ARG, "morphology: op must be 0 (dilation) or 1 (erosion)");
  dim3 blk(32, 8);
  dim3 grid((unsigned)((W + 31) / 32), (unsigned)((H + 7) / 8), (unsigned)(B * Cout));
  morphology_kernel<<<grid, blk, 0, (cudaStream_t)stream>>>(x, weight, out, (int)B, (int)Cin, (int)Cout,
                                                             (int)H, (int)W, ksize, op, soft, beta);
  return check_launch("morphology");
}

}  // extern "C"
