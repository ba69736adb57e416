// Kernels of the LPIPS distance (lpips v0.1, net='vgg'; the regulariser of the masked-prediction guidance,
// src/attr_functions.py apply_lpips) around the tcgen05 convolutions of the VGG-16 trunk: 2x2 stride-2 max pooling
// forward / backward, and the distance head - per-pixel channel normalisation, lin-weighted squared difference against
// the cached normalised features of the reference, spatial mean - with its analytic backward.  Activations are f16 NHWC;
// planes = 3: split tensors [hi | lo | hi] of the fp32-accurate forward (pixel pitch 3 C, value = hi + lo).
#include "unet_kernels.cuh"

namespace b2e {

namespace {
__device__ __forceinline__ void unpack8l(const uint4& v, float* f) {
  const f16x2* b = reinterpret_cast<const f16x2*>(&v);
#pragma unroll
  for (int j = 0; j < 4; ++j) { const float2 t = f16x2_to_float2(b[j]); f[2 * j] = t.x; f[2 * j + 1] = t.y; }
}
__device__ __forceinline__ uint4 pack8l(const float* f) {
  uint4 v;
  f16x2* b = reinterpret_cast<f16x2*>(&v);
#pragma unroll
  for (int j = 0; j < 4; ++j) b[j] = floats_to_f16x2(f[2 * j], f[2 * j + 1]);
  return v;
}
inline int grid_for(int64_t total, int per_sm = 32) {
  int64_t g = (total + 255) / 256;
  if (g > (int64_t)kNumSMs * per_sm) g = (int64_t)kNumSMs * per_sm;
  return (int)(g < 1 ? 1 : g);
}
constexpr float kLpipsEps = 1e-10f;   // lpips.normalize_tensor
}  // namespace

// ---- max pooling 2x2, stride 2 (torch.nn.MaxPool2d(2, 2)): idx = 2 bits per output element, position (dh*2 + dw) of
// the first maximum in scan order; 8 channels per thread -> one uint16 per slot.  planes = 3: candidates are compared on
// hi + lo and both planes of the winner are copied
__global__ void __launch_bounds__(256) maxpool2x2_kernel(const f16* __restrict__ x, f16* __restrict__ y,
                                                         uint16_t* __restrict__ idx, int N, int H, int W, int C8, int planes) {
  pdl_wait();
  const int Ho = H / 2, Wo = W / 2;
  const int64_t total = (int64_t)N * Ho * Wo * C8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(i % C8);
    int64_t r = i / C8;
    const int ow = (int)(r % Wo); r /= Wo;
    const int oh = (int)(r % Ho);
    const int n = (int)(r / Ho);
    float best[8], bhi[8], blo[8];
    uint32_t arg = 0;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const f16* xp = x + ((((int64_t)n * H + 2 * oh + (t >> 1)) * W + 2 * ow + (t & 1)) * (planes * C8) + s) * 8;
      float hi[8], lo[8];
      unpack8l(__ldg(reinterpret_cast<const uint4*>(xp)), hi);
      if (planes == 3) unpack8l(__ldg(reinterpret_cast<const uint4*>(xp + C8 * 8)), lo);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float v = planes == 3 ? hi[j] + lo[j] : hi[j];
        if (t == 0 || v > best[j]) {
          best[j] = v; bhi[j] = hi[j]; blo[j] = planes == 3 ? lo[j] : 0.f;
          arg = (arg & ~(3u << (2 * j))) | ((uint32_t)t << (2 * j));
        }
      }
    }
    if (planes == 1) {
      *reinterpret_cast<uint4*>(y + i * 8) = pack8l(bhi);
    } else {
      f16* o = y + ((i / C8) * (int64_t)(3 * C8) + s) * 8;
      const uint4 hv = pack8l(bhi);      // f16 values: the conversion back is exact
      *reinterpret_cast<uint4*>(o) = hv;
      *reinterpret_cast<uint4*>(o + C8 * 8) = pack8l(blo);
      *reinterpret_cast<uint4*>(o + 2 * C8 * 8) = hv;
    }
    idx[i] = (uint16_t)arg;
  }
}

int maxpool2x2_launch(const f16* x, f16* y, uint16_t* idx, int N, int H, int W, int C, cudaStream_t st, int planes) {
  B2E_REQUIRE(C % 8 == 0 && H % 2 == 0 && W % 2 == 0 && (planes == 1 || planes == 3), B2E_UNSUPPORTED_SHAPE,
              "maxpool2x2: bad shape");
  const int64_t total = (int64_t)N * (H / 2) * (W / 2) * (C / 8);
  launch_pdl(maxpool2x2_kernel, dim3(grid_for(total)), dim3(256), 0, st, x, y, idx, N, H, W, C / 8, planes);
  return check_launch("maxpool2x2");
}

// gx[p] = (x[p] > 0) * (gy[window of p] if p is the window's recorded arg-max else 0); x = the pooled (ReLU) activation
__global__ void __launch_bounds__(256) maxpool2x2_bwd_kernel(const f16* __restrict__ x, const uint16_t* __restrict__ idx,
                                                             const f16* __restrict__ gy, f16* __restrict__ gx, int N, int H,
                                                             int W, int C8, int xplanes) {
  pdl_wait();
  const int Ho = H / 2, Wo = W / 2;
  const int64_t total = (int64_t)N * H * W * C8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(i % C8);
    int64_t r = i / C8;
    const int iw = (int)(r % W); r /= W;
    const int ih = (int)(r % H);
    const int n = (int)(r / H);
    const int64_t o = (((int64_t)n * Ho + (ih >> 1)) * Wo + (iw >> 1)) * C8 + s;
    const uint32_t a = __ldg(idx + o);
    const uint32_t t = (uint32_t)((ih & 1) * 2 + (iw & 1));
    float g[8], xv[8];
    unpack8l(__ldg(reinterpret_cast<const uint4*>(gy) + o), g);
    const f16* xp = x + ((i / C8) * (int64_t)(xplanes * C8) + s) * 8;
    unpack8l(__ldg(reinterpret_cast<const uint4*>(xp)), xv);
    if (xplanes == 3) {
      float l[8];
      unpack8l(__ldg(reinterpret_cast<const uint4*>(xp + C8 * 8)), l);
#pragma unroll
      for (int j = 0; j < 8; ++j) xv[j] += l[j];
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) g[j] = (((a >> (2 * j)) & 3u) == t && xv[j] > 0.f) ? g[j] : 0.f;
    *reinterpret_cast<uint4*>(gx + i * 8) = pack8l(g);
  }
}

int maxpool2x2_bwd_launch(const f16* x, const uint16_t* idx, const f16* gy, f16* gx, int N, int H, int W, int C, cudaStream_t st,
                          int xplanes) {
  B2E_REQUIRE(C % 8 == 0 && H % 2 == 0 && W % 2 == 0, B2E_UNSUPPORTED_SHAPE, "maxpool2x2_bwd: bad shape");
  const int64_t total = (int64_t)N * H * W * (C / 8);
  launch_pdl(maxpool2x2_bwd_kernel, dim3(grid_for(total)), dim3(256), 0, st, x, idx, gy, gx, N, H, W, C / 8, xplanes);
  return check_launch("maxpool2x2_bwd");
}

// ---- distance head.  A group of LP = min(32, C / 8) lanes owns one pixel; every lane holds NCH (1 or 2) 8-channel
// chunks of it.  The pixel loop is uniform across the block (invalid pixels contribute zeros) so that the shuffles of a
// warp always run with all 32 lanes.
namespace {
template <int NCH>
__device__ __forceinline__ void load_feat(const f16* __restrict__ x, int64_t pix, int C, int planes, int lane_g, int LP,
                                          bool valid, float* f) {
#pragma unroll
  for (int c = 0; c < NCH; ++c) {
    const int ch = (c * LP + lane_g) * 8;
    if (valid) {
      const f16* xp = x + pix * (int64_t)(planes * C) + ch;
      unpack8l(__ldg(reinterpret_cast<const uint4*>(xp)), f + 8 * c);
      if (planes == 3) {
        float l[8];
        unpack8l(__ldg(reinterpret_cast<const uint4*>(xp + C)), l);
#pragma unroll
        for (int j = 0; j < 8; ++j) f[8 * c + j] += l[j];
      }
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) f[8 * c + j] = 0.f;
    }
  }
}
__device__ __forceinline__ float group_sum(float v, int LP) {
  for (int o = LP >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
}  // namespace

// mode 0 (reference pass): ref[b][p][c] = f / (||f|| + eps) in fp32.
// mode 1 (distance): partial[b][slot0 + block] = sum over the block's pixels of sum_c w[c] (u0[c] - u1[c])^2 (fp64; fixed
// pixel order per group, fixed order over the groups), u1 = ref[rb][p] with rb = ref_batched ? b : 0.  Also
// hmax[b] = max(hmax[b], max |d/df| of the tap's head gradient for d_dist[b] = 1, after the ReLU mask): the backward's
// gradient scale then accounts for the 1 / ||f|| of the normalisation Jacobian (order-independent max: deterministic).
template <int NCH>
__global__ void __launch_bounds__(256) lpips_head_kernel(const f16* __restrict__ x, int C, int HW, int planes, const float* __restrict__ w,
                                                         float* __restrict__ ref, int ref_batched, double* __restrict__ partial,
                                                         int part_pitch, int slot0, int mode, float* __restrict__ hmax) {
  pdl_wait();
  __shared__ double s_d[256];
  const int LP = C / 8 / NCH, groups = 256 / LP;
  const int g = threadIdx.x / LP, lg = threadIdx.x % LP;
  const int b = blockIdx.y;
  const int64_t img = (int64_t)b * HW;
  const float* rimg = ref + (int64_t)(ref_batched ? b : 0) * HW * C;
  float wv[8 * NCH];
  if (mode == 1) {
#pragma unroll
    for (int c = 0; c < NCH; ++c)
#pragma unroll
      for (int j = 0; j < 8; ++j) wv[8 * c + j] = __ldg(w + (c * LP + lg) * 8 + j);
  }
  double acc = 0.0;
  float hm = 0.f;
  for (int base = blockIdx.x * groups; base < HW; base += gridDim.x * groups) {
    const int p = base + g;
    const bool valid = p < HW;
    float f[8 * NCH];
    load_feat<NCH>(x, img + p, C, planes, lg, LP, valid, f);
    float s2 = 0.f;
#pragma unroll
    for (int j = 0; j < 8 * NCH; ++j) s2 += f[j] * f[j];
    s2 = group_sum(s2, LP);
    const float den = sqrtf(s2) + kLpipsEps;
    if (mode == 0) {
      if (valid) {
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          float u[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) u[j] = __fdiv_rn(f[8 * c + j], den);
          float4* dst = reinterpret_cast<float4*>(ref + (img + p) * C + (c * LP + lg) * 8);
          dst[0] = make_float4(u[0], u[1], u[2], u[3]);
          dst[1] = make_float4(u[4], u[5], u[6], u[7]);
        }
      }
    } else {
      float d = 0.f, fg = 0.f, gt[8 * NCH];
      const float coef = 2.f / (float)HW;
#pragma unroll
      for (int j = 0; j < 8 * NCH; ++j) gt[j] = 0.f;
      if (valid) {
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          const float4* src = reinterpret_cast<const float4*>(rimg + (int64_t)p * C + (c * LP + lg) * 8);
          const float4 r0 = __ldg(src), r1 = __ldg(src + 1);
          const float u1[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float e = __fdiv_rn(f[8 * c + j], den) - u1[j];
            d += wv[8 * c + j] * (e * e);
            gt[8 * c + j] = coef * wv[8 * c + j] * e;
            fg += f[8 * c + j] * gt[8 * c + j];
          }
        }
      }
      d = group_sum(d, LP);
      fg = group_sum(fg, LP);
      acc += (double)d;
      const float s = sqrtf(s2), k = 1.f / den;
      if (valid && s > 0.f) {
        const float t = k * k * fg / s;
#pragma unroll
        for (int j = 0; j < 8 * NCH; ++j)
          if (f[j] > 0.f) hm = fmaxf(hm, fabsf(k * gt[j] - t * f[j]));
      }
    }
  }
  if (mode == 0) return;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) hm = fmaxf(hm, __shfl_xor_sync(0xffffffffu, hm, o));
  // non-negative floats order like their bit patterns (a NaN / inf sorts above every finite value)
  if ((threadIdx.x & 31) == 0 && hm > 0.f) atomicMax(reinterpret_cast<unsigned*>(hmax + b), __float_as_uint(hm));
  if (lg == 0) s_d[g] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < groups; ++i) t += s_d[i];
    partial[(int64_t)b * part_pitch + slot0 + blockIdx.x] = t;
  }
}

int lpips_head_blocks(int HW) {
  int n = (HW + 2047) / 2048;      // ~2048 pixels per block; fixed by the shape (the reduction order depends on it)
  return n < 1 ? 1 : (n > 256 ? 256 : n);
}

int lpips_head_launch(const f16* x, int B, int C, int HW, int planes, const float* w, float* ref, int ref_batched, double* partial,
                      int part_pitch, int slot0, int mode, float* hmax, cudaStream_t st) {
  B2E_REQUIRE(C == 64 || C == 128 || C == 256 || C == 512, B2E_UNSUPPORTED_SHAPE, "lpips_head: %d channels", C);
  const dim3 grid(lpips_head_blocks(HW), B);
  if (C == 512) launch_pdl(lpips_head_kernel<2>, grid, dim3(256), 0, st, x, C, HW, planes, w, ref, ref_batched, partial, part_pitch, slot0, mode, hmax);
  else launch_pdl(lpips_head_kernel<1>, grid, dim3(256), 0, st, x, C, HW, planes, w, ref, ref_batched, partial, part_pitch, slot0, mode, hmax);
  return check_launch("lpips_head");
}

// dist[b] = sum over the five taps of (sum of the tap's partials, in slot order) / HW_tap
__global__ void lpips_finalize_kernel(const double* __restrict__ partial, int part_pitch, LpipsTaps taps, float* __restrict__ dist, int B) {
  pdl_wait();
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  double tot = 0.0;
  for (int k = 0; k < 5; ++k) {
    double s = 0.0;
    for (int i = 0; i < taps.n[k]; ++i) s += partial[(int64_t)b * part_pitch + taps.off[k] + i];
    tot += s / (double)taps.hw[k];
  }
  dist[b] = (float)tot;
}

int lpips_finalize_launch(const double* partial, int part_pitch, const LpipsTaps& taps, float* dist, int B, cudaStream_t st) {
  launch_pdl(lpips_finalize_kernel, dim3((B + 127) / 128), dim3(128), 0, st, partial, part_pitch, taps, dist, B);
  return check_launch("lpips_finalize");
}

// ---- gradient scale of the backward chain: prod[b] = |d_dist[b]| * hmax[b] (the largest head-gradient element of image
// b), then grad_scale_launch puts max_b prod[b] in [2^T, 2^(T+1)) - exact powers of two, as for the other backward passes
__global__ void lpips_grad_bound_kernel(const float* __restrict__ d_dist, const float* __restrict__ hmax, float* __restrict__ prod, int B) {
  pdl_wait();
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < B) prod[b] = fabsf(d_dist[b]) * hmax[b];
}

int lpips_grad_scale_launch(const float* d_dist, const float* hmax, float* prod, int B, float* gs, cudaStream_t st) {
  launch_pdl(lpips_grad_bound_kernel, dim3((B + 127) / 128), dim3(128), 0, st, d_dist, hmax, prod, B);
  int rc = check_launch("lpips_grad_bound");
  if (rc) return rc;
  return grad_scale_launch(prod, B, gs, 1.f, st);
}

// ---- head backward.  s = ||f||, k = 1 / (s + eps), u0 = k f, g = 2 w (u0 - u1) d_dist[b] / HW:
//   d/df = k g - k^2 (f.g) / s f        (fp32; 0 where s = 0)
// then + the gradient arriving from the pooled path (gp, already scaled), ReLU mask of the tap, x gs[0], f16 store.
// The mask is applied BEFORE the f16 store: on an all-zero pixel the exact Jacobian is I / eps.
template <int NCH>
__global__ void __launch_bounds__(256) lpips_head_bwd_kernel(const f16* __restrict__ x, int C, int HW, int planes, const float* __restrict__ w,
                                                             const float* __restrict__ ref, int ref_batched, const float* __restrict__ d_dist,
                                                             const float* __restrict__ gs, const f16* __restrict__ gp, f16* __restrict__ gout,
                                                             int B) {
  pdl_wait();
  const int LP = C / 8 / NCH, groups = 256 / LP;
  const int g = threadIdx.x / LP, lg = threadIdx.x % LP;
  const float sc = gs ? gs[0] : 1.f;
  float wv[8 * NCH];
#pragma unroll
  for (int c = 0; c < NCH; ++c)
#pragma unroll
    for (int j = 0; j < 8; ++j) wv[8 * c + j] = __ldg(w + (c * LP + lg) * 8 + j);
  const int64_t total = (int64_t)B * HW;
  const int64_t stride = (int64_t)gridDim.x * groups;
  for (int64_t base = (int64_t)blockIdx.x * groups; base < total; base += stride) {
    const int64_t pix = base + g;
    const bool valid = pix < total;
    const int b = valid ? (int)(pix / HW) : 0;
    const int p = valid ? (int)(pix - (int64_t)b * HW) : 0;
    float f[8 * NCH];
    load_feat<NCH>(x, pix, C, planes, lg, LP, valid, f);
    float s2 = 0.f;
#pragma unroll
    for (int j = 0; j < 8 * NCH; ++j) s2 += f[j] * f[j];
    s2 = group_sum(s2, LP);
    const float s = sqrtf(s2), den = s + kLpipsEps;
    const float coef = valid ? 2.f * __ldg(d_dist + b) / (float)HW : 0.f;
    float gv[8 * NCH];
    float fg = 0.f;
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      float u1[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if (valid) {
        const float4* src = reinterpret_cast<const float4*>(ref + ((int64_t)(ref_batched ? b : 0) * HW + p) * C + (c * LP + lg) * 8);
        const float4 r0 = __ldg(src), r1 = __ldg(src + 1);
        u1[0] = r0.x; u1[1] = r0.y; u1[2] = r0.z; u1[3] = r0.w; u1[4] = r1.x; u1[5] = r1.y; u1[6] = r1.z; u1[7] = r1.w;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float e = __fdiv_rn(f[8 * c + j], den) - u1[j];
        gv[8 * c + j] = coef * wv[8 * c + j] * e;
        fg += f[8 * c + j] * gv[8 * c + j];
      }
    }
    fg = group_sum(fg, LP);
    if (!valid) continue;
    const float k = 1.f / den;
    const float t = s > 0.f ? k * k * fg / s : 0.f;
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const int64_t off = pix * C + (c * LP + lg) * 8;
      float add[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if (gp) unpack8l(__ldg(reinterpret_cast<const uint4*>(gp + off)), add);
      float o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float v = f[8 * c + j];
        const float dh = s > 0.f ? k * gv[8 * c + j] - t * v : 0.f;
        o[j] = v > 0.f ? dh * sc + add[j] : 0.f;
      }
      *reinterpret_cast<uint4*>(gout + off) = pack8l(o);
    }
  }
}

int lpips_head_bwd_launch(const f16* x, int B, int C, int HW, int planes, const float* w, const float* ref, int ref_batched,
                          const float* d_dist, const float* gs, const f16* gp, f16* gout, cudaStream_t st) {
  B2E_REQUIRE(C == 64 || C == 128 || C == 256 || C == 512, B2E_UNSUPPORTED_SHAPE, "lpips_head_bwd: %d channels", C);
  const int groups = 256 / (C == 512 ? 32 : C / 8);
  int64_t blocks = ((int64_t)B * HW + groups - 1) / groups;
  if (blocks > (int64_t)kNumSMs * 16) blocks = (int64_t)kNumSMs * 16;
  if (C == 512)
    launch_pdl(lpips_head_bwd_kernel<2>, dim3((unsigned)blocks), dim3(256), 0, st, x, C, HW, planes, w, ref, ref_batched, d_dist, gs, gp, gout, B);
  else
    launch_pdl(lpips_head_bwd_kernel<1>, dim3((unsigned)blocks), dim3(256), 0, st, x, C, HW, planes, w, ref, ref_batched, d_dist, gs, gp, gout, B);
  return check_launch("lpips_head_bwd");
}

// ---- guidance: colour gradient of the masked prediction + lam_scale x the LPIPS input gradient (one pass)
__global__ void __launch_bounds__(256) lpips_guidance_grad_kernel(const float* __restrict__ img, const float* __restrict__ mask,
                                                                  const float* __restrict__ d_lp, float* __restrict__ out, int64_t n,
                                                                  int64_t HW, int C, int64_t mask_n, b2e_color_grad_params p) {
  pdl_wait();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)((i / HW) % C);
    const float m = __ldg(mask + i % mask_n);
    float g = 0.f;
    if (p.has_target[c]) g = __fmul_rn(m, p.k[c] * sign_torch(__fmul_rn(m, __ldg(img + i)) - p.target[c]));
    out[i] = g + p.lam_scale * __ldg(d_lp + i);
  }
}

}  // namespace b2e

extern "C" int b2e_lpips_guidance_grad_f32(const float* img, const float* mask, const float* d_lpips, float* d_img, int64_t B,
                                           int64_t C, int64_t HW, const b2e_color_grad_params* p, void* stream) {
  using namespace b2e;
  B2E_REQUIRE(img && mask && d_lpips && d_img && p, B2E_INVALID_ARG, "lpips_guidance_grad: null pointer");
  B2E_REQUIRE(B >= 1 && C >= 1 && C <= 4 && HW >= 1, B2E_UNSUPPORTED_SHAPE, "lpips_guidance_grad: 1..4 channels");
  const int64_t n = B * C * HW;
  launch_pdl(lpips_guidance_grad_kernel, dim3(grid_for(n)), dim3(256), 0, (cudaStream_t)stream, img, mask, d_lpips, d_img, n, HW,
             (int)C, p->mask_batched ? n : C * HW, *p);
  return check_launch("lpips_guidance_grad");
}
