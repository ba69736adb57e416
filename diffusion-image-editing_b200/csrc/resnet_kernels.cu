// Kernels around the tcgen05 convolutions of the classifier network of ClassifierAttrFunc (torchvision ResNet,
// src/models.py:69-77, src/attr_functions.py:222-257): stem im2col (7x7 stride 2) and its col2im gradient, 3x3 stride-2
// max pooling forward / backward, ReLU backward, stride-2 subsampling / zero insertion (stride-2 convolution gradients),
// global average pooling + fully connected head forward / backward.  Activations are f16 NHWC, BatchNorm (eval) is
// folded into the convolution weights and biases by the host, ReLU is fused into the convolution epilogue.
#include "unet_kernels.cuh"

namespace b2e {

namespace {
__device__ __forceinline__ void unpack8r(const uint4& v, float* f) {
  const f16x2* b = reinterpret_cast<const f16x2*>(&v);
#pragma unroll
  for (int j = 0; j < 4; ++j) { const float2 t = f16x2_to_float2(b[j]); f[2 * j] = t.x; f[2 * j + 1] = t.y; }
}
__device__ __forceinline__ uint4 pack8r(const float* f) {
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
}  // namespace

// ---- stem: x fp32 NCHW (B,C,H,W) -> f16 (B,H/2,W/2,KP): column (kh*7 + kw)*C + c = x[c][2oh + kh - 3][2ow + kw - 3]
// planes = 3 (fp32-accurate forward): the pixel holds three KP-column planes [hi | lo | hi], hi = f16(v), lo = f16(v - hi)
__global__ void __launch_bounds__(256) im2col7s2_kernel(const float* __restrict__ x, f16* __restrict__ out, int B, int C, int H,
                                                        int W, int KP, int planes) {
  pdl_wait();
  const int Ho = H / 2, Wo = W / 2, slots = KP / 8, cols = 49 * C;
  const int64_t total = (int64_t)B * Ho * Wo * slots;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(i % slots);
    int64_t r = i / slots;
    const int ow = (int)(r % Wo); r /= Wo;
    const int oh = (int)(r % Ho);
    const int b = (int)(r / Ho);
    float f[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int col = s * 8 + j;
      float v = 0.f;
      if (col < cols) {
        const int t = col / C, c = col - t * C;
        const int ih = 2 * oh + t / 7 - 3, iw = 2 * ow + t % 7 - 3;
        if (ih >= 0 && ih < H && iw >= 0 && iw < W) v = __ldg(x + (((int64_t)b * C + c) * H + ih) * W + iw);
      }
      f[j] = v;
    }
    if (planes == 1) {
      *reinterpret_cast<uint4*>(out + i * 8) = pack8r(f);
    } else {
      f16* o = out + (i / slots) * (int64_t)(3 * KP) + s * 8;
      const uint4 hi = pack8r(f);
      float hf[8];
      unpack8r(hi, hf);
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = __fsub_rn(f[j], hf[j]);
      *reinterpret_cast<uint4*>(o) = hi;
      *reinterpret_cast<uint4*>(o + KP) = pack8r(f);
      *reinterpret_cast<uint4*>(o + 2 * KP) = hi;
    }
  }
}

int im2col7s2_launch(const float* x, f16* out, int B, int C, int H, int W, int KP, cudaStream_t st, int planes) {
  B2E_REQUIRE(49 * C <= KP && KP % 64 == 0 && H % 2 == 0 && W % 2 == 0, B2E_UNSUPPORTED_SHAPE, "im2col7s2: bad shape");
  const int64_t total = (int64_t)B * (H / 2) * (W / 2) * (KP / 8);
  launch_pdl(im2col7s2_kernel, dim3(grid_for(total)), dim3(256), 0, st, x, out, B, C, H, W, KP, planes);
  return check_launch("im2col7s2");
}

// gradient of the stem w.r.t. the image: dx[b][c][ih][iw] = sum over taps with 2oh + kh - 3 = ih, 2ow + kw - 3 = iw of
// dcols[b][oh][ow][(kh*7 + kw)*C + c]; dcols f16 (B,H/2,W/2,KP), dx fp32 NCHW
__global__ void __launch_bounds__(256) col2im7s2_kernel(const f16* __restrict__ dcols, float* __restrict__ dx, int B, int C,
                                                        int H, int W, int KP, const float* __restrict__ gs) {
  pdl_wait();
  const float unscale = gs ? gs[1] : 1.f;
  const int Ho = H / 2, Wo = W / 2;
  const int64_t total = (int64_t)B * H * W;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int iw = (int)(i % W);
    const int ih = (int)((i / W) % H);
    const int b = (int)(i / ((int64_t)W * H));
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int kh = (ih + 3) & 1; kh < 7; kh += 2) {
      const int oh = (ih + 3 - kh) >> 1;
      if (oh < 0 || oh >= Ho) continue;
      for (int kw = (iw + 3) & 1; kw < 7; kw += 2) {
        const int ow = (iw + 3 - kw) >> 1;
        if (ow < 0 || ow >= Wo) continue;
        const f16* p = dcols + (((int64_t)b * Ho + oh) * Wo + ow) * KP + (kh * 7 + kw) * C;
        for (int c = 0; c < C; ++c) acc[c] += f16_to_float(p[c]);
      }
    }
    for (int c = 0; c < C; ++c) dx[(((int64_t)b * C + c) * H + ih) * W + iw] = acc[c] * unscale;
  }
}

int col2im7s2_launch(const f16* dcols, float* dx, int B, int C, int H, int W, int KP, cudaStream_t st, const float* gs) {
  B2E_REQUIRE(C >= 1 && C <= 4 && 49 * C <= KP, B2E_UNSUPPORTED_SHAPE, "col2im7s2: bad shape");
  launch_pdl(col2im7s2_kernel, dim3(grid_for((int64_t)B * H * W)), dim3(256), 0, st, dcols, dx, B, C, H, W, KP, gs);
  return check_launch("col2im7s2");
}

// ---- max pooling 3x3, stride 2, padding 1 (f16 NHWC); idx = position (kh*3 + kw) of the first maximum (scan order)
// planes = 3: x and y are split tensors [hi | lo | hi] (pixel pitch 3 C); candidates are compared on hi + lo
__global__ void __launch_bounds__(256) maxpool3s2_kernel(const f16* __restrict__ x, f16* __restrict__ y,
                                                         uint8_t* __restrict__ idx, int N, int H, int W, int C8, int planes) {
  pdl_wait();
  const int Ho = H / 2, Wo = W / 2;
  const int64_t total = (int64_t)N * Ho * Wo * C8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(i % C8);
    int64_t r = i / C8;
    const int ow = (int)(r % Wo); r /= Wo;
    const int oh = (int)(r % Ho);
    const int n = (int)(r / Ho);
    float best[8];
    uint8_t arg[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { best[j] = -INFINITY; arg[j] = 0; }
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      const int ih = 2 * oh + t / 3 - 1, iw = 2 * ow + t % 3 - 1;
      if (ih < 0 || ih >= H || iw < 0 || iw >= W) continue;
      float f[8];
      const f16* xp = x + ((((int64_t)n * H + ih) * W + iw) * (planes * C8) + s) * 8;
      unpack8r(__ldg(reinterpret_cast<const uint4*>(xp)), f);
      if (planes == 3) {
        float l[8];
        unpack8r(__ldg(reinterpret_cast<const uint4*>(xp + C8 * 8)), l);
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] += l[j];
      }
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (f[j] > best[j]) { best[j] = f[j]; arg[j] = (uint8_t)t; }
    }
    if (planes == 1) {
      *reinterpret_cast<uint4*>(y + i * 8) = pack8r(best);
    } else {
      f16* o = y + ((i / C8) * (int64_t)(3 * C8) + s) * 8;
      const uint4 hi = pack8r(best);
      float hf[8];
      unpack8r(hi, hf);
#pragma unroll
      for (int j = 0; j < 8; ++j) hf[j] = __fsub_rn(best[j], hf[j]);
      *reinterpret_cast<uint4*>(o) = hi;
      *reinterpret_cast<uint4*>(o + C8 * 8) = pack8r(hf);
      *reinterpret_cast<uint4*>(o + 2 * C8 * 8) = hi;
    }
    uint2 a;
    a.x = arg[0] | (arg[1] << 8) | (arg[2] << 16) | ((uint32_t)arg[3] << 24);
    a.y = arg[4] | (arg[5] << 8) | (arg[6] << 16) | ((uint32_t)arg[7] << 24);
    *reinterpret_cast<uint2*>(idx + i * 8) = a;
  }
}

int maxpool3s2_launch(const f16* x, f16* y, uint8_t* idx, int N, int H, int W, int C, cudaStream_t st, int planes) {
  B2E_REQUIRE(C % 8 == 0 && H % 2 == 0 && W % 2 == 0, B2E_UNSUPPORTED_SHAPE, "maxpool: bad shape");
  const int64_t total = (int64_t)N * (H / 2) * (W / 2) * (C / 8);
  launch_pdl(maxpool3s2_kernel, dim3(grid_for(total)), dim3(256), 0, st, x, y, idx, N, H, W, C / 8, planes);
  return check_launch("maxpool3s2");
}

// gx[p] = (x[p] > 0) * sum over the (<= 4) windows whose recorded argmax is p of gy[window]   (the x > 0 factor is the
// backward of the ReLU that produced x)
__global__ void __launch_bounds__(256) maxpool3s2_bwd_kernel(const f16* __restrict__ x, const uint8_t* __restrict__ idx,
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
    float acc[8], xv[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    {
      const f16* xp = x + ((i / C8) * (int64_t)(xplanes * C8) + s) * 8;     // forward activation: split tensor when xplanes = 3
      unpack8r(__ldg(reinterpret_cast<const uint4*>(xp)), xv);
      if (xplanes == 3) {
        float l[8];
        unpack8r(__ldg(reinterpret_cast<const uint4*>(xp + C8 * 8)), l);
#pragma unroll
        for (int j = 0; j < 8; ++j) xv[j] += l[j];
      }
    }
    // windows oh with 2*oh - 1 <= ih <= 2*oh + 1
    for (int oh = ih >> 1; oh <= ((ih + 1) >> 1); ++oh) {
      if (oh >= Ho) continue;
      const int kh = ih - (2 * oh - 1);
      for (int ow = iw >> 1; ow <= ((iw + 1) >> 1); ++ow) {
        if (ow >= Wo) continue;
        const int t = kh * 3 + (iw - (2 * ow - 1));
        const int64_t o = ((((int64_t)n * Ho + oh) * Wo + ow) * C8 + s) * 8;
        const uint2 a = __ldg(reinterpret_cast<const uint2*>(idx + o));
        float g[8];
        unpack8r(__ldg(reinterpret_cast<const uint4*>(gy + o)), g);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint32_t aj = ((j < 4 ? a.x : a.y) >> (8 * (j & 3))) & 0xffu;
          if ((int)aj == t) acc[j] += g[j];
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = xv[j] > 0.f ? acc[j] : 0.f;
    *reinterpret_cast<uint4*>(gx + i * 8) = pack8r(acc);
  }
}

int maxpool3s2_bwd_launch(const f16* x, const uint8_t* idx, const f16* gy, f16* gx, int N, int H, int W, int C,
                          cudaStream_t st, int xplanes) {
  const int64_t total = (int64_t)N * H * W * (C / 8);
  launch_pdl(maxpool3s2_bwd_kernel, dim3(grid_for(total)), dim3(256), 0, st, x, idx, gy, gx, N, H, W, C / 8, xplanes);
  return check_launch("maxpool3s2_bwd");
}

// ---- ReLU backward: out = g * (y > 0)   (out may alias g)
__global__ void __launch_bounds__(256) relu_bwd_kernel(const uint4* __restrict__ g, const uint4* __restrict__ y,
                                                       uint4* __restrict__ out, int64_t n8) {
  pdl_wait();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
    float gv[8], yv[8];
    unpack8r(g[i], gv);
    unpack8r(__ldg(y + i), yv);
#pragma unroll
    for (int j = 0; j < 8; ++j) gv[j] = yv[j] > 0.f ? gv[j] : 0.f;
    out[i] = pack8r(gv);
  }
}

// the same with y a split tensor [hi | lo | hi] of the fp32-accurate forward (pixel pitch 3 C): mask = (hi + lo > 0)
__global__ void __launch_bounds__(256) relu_bwd_split_kernel(const uint4* __restrict__ g, const uint4* __restrict__ y,
                                                             uint4* __restrict__ out, int64_t n8, int C8) {
  pdl_wait();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / C8;
    const int s = (int)(i - row * C8);
    float gv[8], yv[8], lv[8];
    unpack8r(g[i], gv);
    unpack8r(__ldg(y + row * 3 * C8 + s), yv);
    unpack8r(__ldg(y + row * 3 * C8 + C8 + s), lv);
#pragma unroll
    for (int j = 0; j < 8; ++j) gv[j] = (yv[j] + lv[j]) > 0.f ? gv[j] : 0.f;
    out[i] = pack8r(gv);
  }
}

int relu_bwd_launch(const f16* g, const f16* y, f16* out, int64_t numel, cudaStream_t st, int yplanes, int C) {
  B2E_REQUIRE(numel % 8 == 0, B2E_UNSUPPORTED_SHAPE, "relu_bwd: numel %% 8 != 0");
  if (yplanes == 3) {
    B2E_REQUIRE(C > 0 && C % 8 == 0, B2E_UNSUPPORTED_SHAPE, "relu_bwd: split activation needs the channel count");
    launch_pdl(relu_bwd_split_kernel, dim3(grid_for(numel / 8)), dim3(256), 0, st, (const uint4*)g, (const uint4*)y, (uint4*)out,
               numel / 8, C / 8);
    return check_launch("relu_bwd_split");
  }
  launch_pdl(relu_bwd_kernel, dim3(grid_for(numel / 8)), dim3(256), 0, st, (const uint4*)g, (const uint4*)y, (uint4*)out, numel / 8);
  return check_launch("relu_bwd");
}

// ---- stride-2 helpers: subsample (x[:, ::2, ::2]) and its adjoint (zero insertion)
__global__ void __launch_bounds__(256) subsample2x_kernel(const uint4* __restrict__ in, uint4* __restrict__ out, int N, int Ho,
                                                          int Wo, int C8) {
  pdl_wait();
  const int64_t total = (int64_t)N * Ho * Wo * C8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C8);
    int64_t r = i / C8;
    const int ow = (int)(r % Wo); r /= Wo;
    const int oh = (int)(r % Ho);
    const int n = (int)(r / Ho);
    out[i] = __ldg(in + (((int64_t)n * 2 * Ho + 2 * oh) * 2 * Wo + 2 * ow) * C8 + c);
  }
}

int subsample2x_launch(const f16* in, f16* out, int N, int Ho, int Wo, int C, cudaStream_t st) {
  B2E_REQUIRE(C % 8 == 0, B2E_UNSUPPORTED_SHAPE, "subsample: C %% 8 != 0");
  launch_pdl(subsample2x_kernel, dim3(grid_for((int64_t)N * Ho * Wo * (C / 8))), dim3(256), 0, st, (const uint4*)in, (uint4*)out,
             N, Ho, Wo, C / 8);
  return check_launch("subsample2x");
}

__global__ void __launch_bounds__(256) zero_upsample2x_kernel(const uint4* __restrict__ in, uint4* __restrict__ out, int N,
                                                              int Hi, int Wi, int C8) {
  pdl_wait();
  const int64_t total = (int64_t)N * 4 * Hi * Wi * C8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C8);
    int64_t r = i / C8;
    const int w = (int)(r % (2 * Wi)); r /= (2 * Wi);
    const int h = (int)(r % (2 * Hi));
    const int n = (int)(r / (2 * Hi));
    uint4 v = make_uint4(0, 0, 0, 0);
    if (!(h & 1) && !(w & 1)) v = __ldg(in + (((int64_t)n * Hi + (h >> 1)) * Wi + (w >> 1)) * C8 + c);
    out[i] = v;
  }
}

int zero_upsample2x_launch(const f16* in, f16* out, int N, int Hi, int Wi, int C, cudaStream_t st) {
  B2E_REQUIRE(C % 8 == 0, B2E_UNSUPPORTED_SHAPE, "zero_upsample: C %% 8 != 0");
  launch_pdl(zero_upsample2x_kernel, dim3(grid_for((int64_t)N * 4 * Hi * Wi * (C / 8))), dim3(256), 0, st, (const uint4*)in,
             (uint4*)out, N, Hi, Wi, C / 8);
  return check_launch("zero_upsample2x");
}

// ---- head: global average pooling + fully connected layer
__global__ void __launch_bounds__(256) avgpool_kernel(const f16* __restrict__ x, float* __restrict__ feat, int HW, int C,
                                                      int planes) {
  pdl_wait();
  const int n = blockIdx.y, c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float s = 0.f;
  const int P = planes * C;
  if (planes == 3) {
    for (int p = 0; p < HW; ++p) {
      const f16* q = x + ((int64_t)n * HW + p) * P + c;
      s += f16_to_float(q[0]) + f16_to_float(q[C]);
    }
  } else {
    for (int p = 0; p < HW; ++p) s += f16_to_float(x[((int64_t)n * HW + p) * C + c]);
  }
  feat[(int64_t)n * C + c] = s / (float)HW;
}

__global__ void __launch_bounds__(256) fc_kernel(const float* __restrict__ feat, const float* __restrict__ w,
                                                 const float* __restrict__ b, float* __restrict__ out, int N, int C, int K) {
  pdl_wait();
  const int wid = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (wid >= N * K) return;
  const int n = wid / K, k = wid % K;
  float s = 0.f;
  for (int c = lane; c < C; c += 32) s += __ldg(w + (int64_t)k * C + c) * feat[(int64_t)n * C + c];
  s = warp_sum(s);
  if (lane == 0) out[(int64_t)n * K + k] = s + b[k];
}

int avgpool_fc_launch(const f16* x, float* feat, const float* w, const float* b, float* logits, int N, int HW, int C, int K,
                      cudaStream_t st, int planes) {
  launch_pdl(avgpool_kernel, dim3((C + 255) / 256, N), dim3(256), 0, st, x, feat, HW, C, planes);
  int rc = check_launch("avgpool");
  if (rc) return rc;
  launch_pdl(fc_kernel, dim3((N * K + 7) / 8), dim3(256), 0, st, (const float*)feat, w, b, logits, N, C, K);
  return check_launch("fc");
}

// backward of the head: dfeat = W^T dlogits ; g[n][p][c] = (y[n][p][c] > 0) ? dfeat[n][c] / HW : 0   (y = the ReLU output
// the pooling read, so g is already the gradient w.r.t. the last block's pre-activation)
__global__ void __launch_bounds__(256) fc_bwd_kernel(const float* __restrict__ dlogits, const float* __restrict__ w,
                                                     float* __restrict__ dfeat, int C, int K, float scale,
                                                     const float* __restrict__ gs) {
  pdl_wait();
  if (gs) scale *= gs[0];
  const int n = blockIdx.y, c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float s = 0.f;
  for (int k = 0; k < K; ++k) s += dlogits[(int64_t)n * K + k] * __ldg(w + (int64_t)k * C + c);
  dfeat[(int64_t)n * C + c] = s * scale;
}

__global__ void __launch_bounds__(256) avgpool_bwd_kernel(const float* __restrict__ dfeat, const f16* __restrict__ y,
                                                          f16* __restrict__ g, int HW, int C8, int yplanes) {
  pdl_wait();
  const int n = blockIdx.y;
  const int64_t total = (int64_t)HW * C8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(i % C8);
    float yv[8], o[8];
    const f16* yp = y + (((int64_t)n * HW + i / C8) * (yplanes * C8) + s) * 8;
    unpack8r(__ldg(reinterpret_cast<const uint4*>(yp)), yv);
    if (yplanes == 3) {
      float l[8];
      unpack8r(__ldg(reinterpret_cast<const uint4*>(yp + C8 * 8)), l);
#pragma unroll
      for (int j = 0; j < 8; ++j) yv[j] += l[j];
    }
    const float* d = dfeat + (int64_t)n * C8 * 8 + s * 8;
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = yv[j] > 0.f ? d[j] : 0.f;
    *reinterpret_cast<uint4*>(g + ((int64_t)n * total + i) * 8) = pack8r(o);
  }
}

int avgpool_fc_bwd_launch(const float* dlogits, const float* w, float* dfeat, const f16* y, f16* g, int N, int HW, int C, int K,
                          cudaStream_t st, const float* gs, int yplanes) {
  launch_pdl(fc_bwd_kernel, dim3((C + 255) / 256, N), dim3(256), 0, st, dlogits, w, dfeat, C, K, 1.0f / (float)HW, gs);
  int rc = check_launch("fc_bwd");
  if (rc) return rc;
  const int64_t total = (int64_t)HW * (C / 8);
  launch_pdl(avgpool_bwd_kernel, dim3((unsigned)((total + 255) / 256), N), dim3(256), 0, st, (const float*)dfeat, y, g, HW, C / 8, yplanes);
  return check_launch("avgpool_bwd");
}

// ---- face parser (BiSeNet, src/Segmentation/model.py) helpers
int avgpool_launch(const f16* x, float* feat, int N, int HW, int C, cudaStream_t st, int planes) {
  launch_pdl(avgpool_kernel, dim3((C + 255) / 256, N), dim3(256), 0, st, x, feat, HW, C, planes);
  return check_launch("avgpool");
}

// out[n][k] = act(w[k] . x[n] + b[k]); act: 0 none, 1 relu, 2 sigmoid, 3 1 + sigmoid   (1x1 convolutions on pooled vectors)
__global__ void __launch_bounds__(256) fc_act_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                     const float* __restrict__ b, float* __restrict__ out, int N, int C, int K,
                                                     int act) {
  pdl_wait();
  const int wid = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (wid >= N * K) return;
  const int n = wid / K, k = wid % K;
  float s = 0.f;
  for (int c = lane; c < C; c += 32) s += __ldg(w + (int64_t)k * C + c) * x[(int64_t)n * C + c];
  s = warp_sum(s);
  if (lane == 0) {
    if (b) s += b[k];
    if (act == 1) s = fmaxf(s, 0.f);
    else if (act >= 2) s = 1.f / (1.f + expf(-s)) + (act == 3 ? 1.f : 0.f);
    out[(int64_t)n * K + k] = s;
  }
}

int fc_act_launch(const float* x, const float* w, const float* b, float* out, int N, int C, int K, int act, cudaStream_t st) {
  launch_pdl(fc_act_kernel, dim3((N * K + 7) / 8), dim3(256), 0, st, x, w, b, out, N, C, K, act);
  return check_launch("fc_act");
}

// out[n][p][c] = x[n][p][c] * a[n][c] (+ b[n][c]) (+ y[n][p][c])   (channel attention / broadcast add, f16 NHWC)
__global__ void __launch_bounds__(256) chan_affine_kernel(const f16* __restrict__ x, const float* __restrict__ a,
                                                          const float* __restrict__ b, const f16* __restrict__ y,
                                                          f16* __restrict__ out, int HW, int C8, int planes) {
  pdl_wait();
  const int n = blockIdx.y;
  const int64_t total = (int64_t)HW * C8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(i % C8);
    // planes = 3: x, y and out are split tensors [hi | lo | hi] (pixel pitch 3 C): value = hi + lo
    const int64_t o = planes == 1 ? ((int64_t)n * total + i) * 8 : ((((int64_t)n * HW + i / C8) * 3) * C8 + s) * 8;
    float xv[8], yv[8];
    unpack8r(__ldg(reinterpret_cast<const uint4*>(x + o)), xv);
    if (y) unpack8r(__ldg(reinterpret_cast<const uint4*>(y + o)), yv);
    if (planes == 3) {
      float l[8];
      unpack8r(__ldg(reinterpret_cast<const uint4*>(x + o + C8 * 8)), l);
#pragma unroll
      for (int j = 0; j < 8; ++j) xv[j] += l[j];
      if (y) {
        unpack8r(__ldg(reinterpret_cast<const uint4*>(y + o + C8 * 8)), l);
#pragma unroll
        for (int j = 0; j < 8; ++j) yv[j] += l[j];
      }
    }
    const float* ap = a ? a + (int64_t)n * C8 * 8 + s * 8 : nullptr;
    const float* bp = b ? b + (int64_t)n * C8 * 8 + s * 8 : nullptr;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float v = ap ? xv[j] * ap[j] : xv[j];
      if (bp) v += bp[j];
      if (y) v += yv[j];
      xv[j] = v;
    }
    const uint4 hi = pack8r(xv);
    *reinterpret_cast<uint4*>(out + o) = hi;
    if (planes == 3) {
      float hf[8];
      unpack8r(hi, hf);
#pragma unroll
      for (int j = 0; j < 8; ++j) hf[j] = __fsub_rn(xv[j], hf[j]);
      *reinterpret_cast<uint4*>(out + o + C8 * 8) = pack8r(hf);
      *reinterpret_cast<uint4*>(out + o + 2 * C8 * 8) = hi;
    }
  }
}

int chan_affine_launch(const f16* x, const float* a, const float* b, const f16* y, f16* out, int N, int HW, int C,
                       cudaStream_t st, int planes) {
  B2E_REQUIRE(C % 8 == 0, B2E_UNSUPPORTED_SHAPE, "chan_affine: C %% 8 != 0");
  const int64_t total = (int64_t)HW * (C / 8);
  int gx = (int)((total + 255) / 256);
  if (gx > kNumSMs * 8) gx = kNumSMs * 8;
  launch_pdl(chan_affine_kernel, dim3(gx, N), dim3(256), 0, st, x, a, b, y, out, HW, C / 8, planes);
  return check_launch("chan_affine");
}

// ---- backward helpers of the face parser
// out[n][c] = scale * sum_p x[n][p][c] * (y ? y[n][p][c] : 1)   (gradient of a per-channel attention / broadcast vector)
__global__ void __launch_bounds__(256) chan_dot_kernel(const f16* __restrict__ x, const f16* __restrict__ y,
                                                       float* __restrict__ out, int HW, int C, float scale, int yplanes) {
  pdl_wait();
  __shared__ float red[256];
  const int n = blockIdx.y, c0 = blockIdx.x * 32, lane = threadIdx.x & 31, row = threadIdx.x >> 5;   // 8 pixel rows x 32 channels
  const int c = c0 + lane;
  float s = 0.f;
  if (c < C)
    for (int p = row; p < HW; p += 8) {
      const int64_t o = ((int64_t)n * HW + p) * C + c;
      const float xv = f16_to_float(x[o]);
      if (y) {
        const f16* yp = y + ((int64_t)n * HW + p) * (yplanes * C) + c;     // yplanes = 3: split forward activation, hi + lo
        s += xv * (yplanes == 3 ? f16_to_float(yp[0]) + f16_to_float(yp[C]) : f16_to_float(yp[0]));
      } else {
        s += xv;
      }
    }
  red[threadIdx.x] = s;
  __syncthreads();
  if (row == 0 && c < C) {
    float t = 0.f;
    for (int r = 0; r < 8; ++r) t += red[r * 32 + lane];
    out[(int64_t)n * C + c] = t * scale;
  }
}

int chan_dot_launch(const f16* x, const f16* y, float* out, int N, int HW, int C, float scale, cudaStream_t st, int yplanes) {
  launch_pdl(chan_dot_kernel, dim3((C + 31) / 32, N), dim3(256), 0, st, x, y, out, HW, C, scale, yplanes);
  return check_launch("chan_dot");
}

// out[n][c] = scale * sum_k g[n][k] * w[k][c]   (transposed 1x1 convolution on pooled vectors)
int fc_t_launch(const float* g, const float* w, float* out, int N, int C, int K, float scale, cudaStream_t st) {
  launch_pdl(fc_bwd_kernel, dim3((C + 255) / 256, N), dim3(256), 0, st, g, w, out, C, K, scale, (const float*)nullptr);
  return check_launch("fc_t");
}

// element-wise on [n] vectors: mode 0: out = g * (a > 0) (ReLU), 1: out = g * a * (1 - a) (sigmoid output a),
// 2: out = g * (a - 1) * (2 - a) (a = 1 + sigmoid)
__global__ void __launch_bounds__(256) vec_act_bwd_kernel(const float* __restrict__ g, const float* __restrict__ a,
                                                          float* __restrict__ out, int n, int mode) {
  pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float av = a[i], gv = g[i];
  out[i] = mode == 0 ? (av > 0.f ? gv : 0.f) : mode == 1 ? gv * av * (1.f - av) : gv * (av - 1.f) * (2.f - av);
}

int vec_act_bwd_launch(const float* g, const float* a, float* out, int n, int mode, cudaStream_t st) {
  launch_pdl(vec_act_bwd_kernel, dim3((n + 255) / 256), dim3(256), 0, st, g, a, out, n, mode);
  return check_launch("vec_act_bwd");
}

// out[r][c] = (g[r][c] + e[r * e_pitch + e_off + c]) * (y ? y[r][c] > 0 : 1): gradient accumulation from a second
// consumer (a channel window of a wider tensor) followed by the ReLU mask of the tensor both consumers read
__global__ void __launch_bounds__(256) grad_merge_kernel(const f16* __restrict__ g, const f16* __restrict__ e, int e_pitch,
                                                         int e_off, const f16* __restrict__ y, f16* __restrict__ out,
                                                         int64_t rows, int C8, int yplanes) {
  pdl_wait();
  const int64_t total = rows * C8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(i % C8);
    const int64_t r = i / C8;
    float gv[8], ev[8], yv[8];
    if (g) unpack8r(*reinterpret_cast<const uint4*>(g + i * 8), gv);
    else {
#pragma unroll
      for (int j = 0; j < 8; ++j) gv[j] = 0.f;
    }
    if (e) {
      unpack8r(__ldg(reinterpret_cast<const uint4*>(e + r * e_pitch + e_off + s * 8)), ev);
#pragma unroll
      for (int j = 0; j < 8; ++j) gv[j] += ev[j];
    }
    if (y) {
      const f16* yp = y + (r * (yplanes * C8) + s) * 8;      // yplanes = 3: split forward activation, mask on hi + lo
      unpack8r(__ldg(reinterpret_cast<const uint4*>(yp)), yv);
      if (yplanes == 3) {
        float l[8];
        unpack8r(__ldg(reinterpret_cast<const uint4*>(yp + C8 * 8)), l);
#pragma unroll
        for (int j = 0; j < 8; ++j) yv[j] += l[j];
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) gv[j] = yv[j] > 0.f ? gv[j] : 0.f;
    }
    *reinterpret_cast<uint4*>(out + i * 8) = pack8r(gv);
  }
}

int grad_merge_launch(const f16* g, const f16* e, int e_pitch, int e_off, const f16* y, f16* out, int64_t rows, int C,
                      cudaStream_t st, int yplanes) {
  B2E_REQUIRE(C % 8 == 0 && e_pitch % 8 == 0 && e_off % 8 == 0, B2E_UNSUPPORTED_SHAPE, "grad_merge: alignment");
  launch_pdl(grad_merge_kernel, dim3(grid_for(rows * (C / 8))), dim3(256), 0, st, g, e, e_pitch, e_off, y, out, rows, C / 8, yplanes);
  return check_launch("grad_merge");
}

// adjoint of the align_corners bilinear upsampling: g (N,K,Ho,Wo) fp32 NCHW -> dx f16 NHWC (N,Hi,Wi,P), channels >= K zero
__global__ void __launch_bounds__(128) bilinear_ac_bwd_kernel(const float* __restrict__ g, f16* __restrict__ dx, int N, int Hi,
                                                              int Wi, int P, int K, int Ho, int Wo, float sh, float sw,
                                                              const float* __restrict__ gs) {
  pdl_wait();
  const float sc = gs ? gs[0] : 1.f;
  const int64_t total = (int64_t)N * Hi * Wi * K;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int k = (int)(i % K);
    int64_t r = i / K;
    const int w = (int)(r % Wi); r /= Wi;
    const int h = (int)(r % Hi);
    const int n = (int)(r / Hi);
    // destination rows whose source coordinate sh * oh lies in (h - 1, h + 1)
    const int oh0 = sh > 0.f ? max(0, (int)ceilf((float)(h - 1) / sh)) : 0, oh1 = sh > 0.f ? min(Ho - 1, (int)floorf((float)(h + 1) / sh)) : Ho - 1;
    const int ow0 = sw > 0.f ? max(0, (int)ceilf((float)(w - 1) / sw)) : 0, ow1 = sw > 0.f ? min(Wo - 1, (int)floorf((float)(w + 1) / sw)) : Wo - 1;
    const float* gp = g + ((int64_t)n * K + k) * Ho * Wo;
    float acc = 0.f;
    for (int oh = oh0; oh <= oh1; ++oh) {
      const float fh = sh * (float)oh;
      const int h0 = (int)fh, h1 = h0 + (h0 < Hi - 1 ? 1 : 0);
      const float lh = fh - (float)h0;
      const float wh = (h0 == h ? 1.f - lh : 0.f) + (h1 == h ? lh : 0.f);
      if (wh == 0.f) continue;
      float rowacc = 0.f;
      for (int ow = ow0; ow <= ow1; ++ow) {
        const float fw = sw * (float)ow;
        const int w0 = (int)fw, w1 = w0 + (w0 < Wi - 1 ? 1 : 0);
        const float lw = fw - (float)w0;
        const float ww = (w0 == w ? 1.f - lw : 0.f) + (w1 == w ? lw : 0.f);
        rowacc += ww * __ldg(gp + (int64_t)oh * Wo + ow);
      }
      acc += wh * rowacc;
    }
    dx[(((int64_t)n * Hi + h) * Wi + w) * P + k] = float_to_f16(acc * sc);
  }
}

__global__ void __launch_bounds__(256) zero_tail_kernel(f16* __restrict__ x, int64_t rows, int P, int K) {
  pdl_wait();
  const int64_t total = rows * (P - K);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x)
    x[(i / (P - K)) * P + K + i % (P - K)] = float_to_f16(0.f);
}

int bilinear_ac_bwd_launch(const float* g, f16* dx, int N, int Hi, int Wi, int P, int K, int Ho, int Wo, cudaStream_t st,
                           const float* gs) {
  const float sh = Ho > 1 ? (float)(Hi - 1) / (float)(Ho - 1) : 0.f, sw = Wo > 1 ? (float)(Wi - 1) / (float)(Wo - 1) : 0.f;
  if (P > K) {
    launch_pdl(zero_tail_kernel, dim3(grid_for((int64_t)N * Hi * Wi * (P - K))), dim3(256), 0, st, dx, (int64_t)N * Hi * Wi, P, K);
    int rc = check_launch("zero_tail");
    if (rc) return rc;
  }
  launch_pdl(bilinear_ac_bwd_kernel, dim3(grid_for((int64_t)N * Hi * Wi * K, 64)), dim3(128), 0, st, g, dx, N, Hi, Wi, P, K, Ho, Wo, sh, sw, gs);
  return check_launch("bilinear_ac_bwd");
}

// F.interpolate(x, (Ho, Wo), mode="bilinear", align_corners=True) at one output pixel: the four source pixels and the
// weights.  ATen's arithmetic: src = dst * (in-1)/(out-1); weights (1-l, l).
struct BilinearTap {
  const f16 *p00, *p01, *p10, *p11;
  float lh, lw;
};

__device__ __forceinline__ BilinearTap bilinear_ac_tap(const f16* x, int n, int oh, int ow, int Hi, int Wi, int PP, float sh,
                                                       float sw) {
  const float fh = sh * (float)oh, fw = sw * (float)ow;
  const int h0 = (int)fh, w0 = (int)fw;
  const int h1 = h0 + (h0 < Hi - 1 ? 1 : 0), w1 = w0 + (w0 < Wi - 1 ? 1 : 0);
  BilinearTap t;
  t.lh = fh - (float)h0;
  t.lw = fw - (float)w0;
  t.p00 = x + (((int64_t)n * Hi + h0) * Wi + w0) * PP;
  t.p01 = x + (((int64_t)n * Hi + h0) * Wi + w1) * PP;
  t.p10 = x + (((int64_t)n * Hi + h1) * Wi + w0) * PP;
  t.p11 = x + (((int64_t)n * Hi + h1) * Wi + w1) * PP;
  return t;
}

// Channel k of the upsampled value.  The logits kernel and the label kernel both call this, so a label is the argmax of
// exactly the logits; the roundings are spelled out (they are the contraction the compiler chose for the original
// expression (1-lh)((1-lw) v00 + lw v01) + lh((1-lw) v10 + lw v11)) so that no kernel can contract them differently.
__device__ __forceinline__ float bilinear_ac_value(const BilinearTap& t, int k, int P, int planes) {
  auto val = [&](const f16* q) { return planes == 3 ? __fadd_rn(f16_to_float(q[k]), f16_to_float(q[P + k])) : f16_to_float(q[k]); };
  const float r0 = __fmaf_rn(1.f - t.lw, val(t.p00), __fmul_rn(t.lw, val(t.p01)));
  const float r1 = __fmaf_rn(1.f - t.lw, val(t.p10), __fmul_rn(t.lw, val(t.p11)));
  return __fmaf_rn(1.f - t.lh, r0, __fmul_rn(t.lh, r1));
}

// x f16 NHWC (N,Hi,Wi,P), first K channels -> out fp32 NCHW (N,K,Ho,Wo).  planes = 3: split tensor [hi | lo | hi] per
// pixel, value = hi + lo.
__global__ void __launch_bounds__(256) bilinear_ac_kernel(const f16* __restrict__ x, float* __restrict__ out, int N, int Hi,
                                                          int Wi, int P, int K, int Ho, int Wo, float sh, float sw, int planes) {
  pdl_wait();
  const int64_t total = (int64_t)N * Ho * Wo;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int ow = (int)(i % Wo);
    const int oh = (int)((i / Wo) % Ho);
    const int n = (int)(i / ((int64_t)Wo * Ho));
    const BilinearTap t = bilinear_ac_tap(x, n, oh, ow, Hi, Wi, P * planes, sh, sw);
    for (int k = 0; k < K; ++k) out[(((int64_t)n * K + k) * Ho + oh) * Wo + ow] = bilinear_ac_value(t, k, P, planes);
  }
}

// The same upsampling followed by argmax over the K channels: labels int64 (N,Ho,Wo), no logits in memory.  torch.argmax
// semantics: the first maximum wins a tie, and a NaN is the maximum (the first NaN).
__global__ void __launch_bounds__(256) bilinear_ac_argmax_kernel(const f16* __restrict__ x, int64_t* __restrict__ labels, int N,
                                                                 int Hi, int Wi, int P, int K, int Ho, int Wo, float sh, float sw,
                                                                 int planes) {
  pdl_wait();
  const int64_t total = (int64_t)N * Ho * Wo;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int ow = (int)(i % Wo);
    const int oh = (int)((i / Wo) % Ho);
    const int n = (int)(i / ((int64_t)Wo * Ho));
    const BilinearTap t = bilinear_ac_tap(x, n, oh, ow, Hi, Wi, P * planes, sh, sw);
    float best = bilinear_ac_value(t, 0, P, planes);
    int arg = 0;
    for (int k = 1; k < K && best == best; ++k) {
      const float v = bilinear_ac_value(t, k, P, planes);
      if (v > best || v != v) { best = v; arg = k; }
    }
    labels[i] = arg;
  }
}

static void bilinear_ac_scales(int Hi, int Wi, int Ho, int Wo, float* sh, float* sw) {
  *sh = Ho > 1 ? (float)(Hi - 1) / (float)(Ho - 1) : 0.f;
  *sw = Wo > 1 ? (float)(Wi - 1) / (float)(Wo - 1) : 0.f;
}

int bilinear_ac_launch(const f16* x, float* out, int N, int Hi, int Wi, int P, int K, int Ho, int Wo, cudaStream_t st, int planes) {
  float sh, sw;
  bilinear_ac_scales(Hi, Wi, Ho, Wo, &sh, &sw);
  launch_pdl(bilinear_ac_kernel, dim3(grid_for((int64_t)N * Ho * Wo)), dim3(256), 0, st, x, out, N, Hi, Wi, P, K, Ho, Wo, sh, sw, planes);
  return check_launch("bilinear_ac");
}

int bilinear_ac_argmax_launch(const f16* x, int64_t* labels, int N, int Hi, int Wi, int P, int K, int Ho, int Wo, cudaStream_t st,
                              int planes) {
  float sh, sw;
  bilinear_ac_scales(Hi, Wi, Ho, Wo, &sh, &sw);
  launch_pdl(bilinear_ac_argmax_kernel, dim3(grid_for((int64_t)N * Ho * Wo)), dim3(256), 0, st, x, labels, N, Hi, Wi, P, K, Ho, Wo,
             sh, sw, planes);
  return check_launch("bilinear_ac_argmax");
}

}  // namespace b2e

extern "C" int b2e_bilinear_ac_argmax_f16(const void* x, int64_t* labels, int64_t N, int64_t Hi, int64_t Wi, int64_t P, int64_t K,
                                          int64_t S, int planes, void* stream) {
  B2E_REQUIRE(x && labels, B2E_INVALID_ARG, "bilinear_ac_argmax: null pointer");
  B2E_REQUIRE(N > 0 && Hi > 0 && Wi > 0 && S > 0 && K >= 1 && K <= P, B2E_UNSUPPORTED_SHAPE, "bilinear_ac_argmax: bad shape");
  B2E_REQUIRE(planes == 1 || planes == 3, B2E_INVALID_ARG, "bilinear_ac_argmax: planes must be 1 or 3");
  return b2e::bilinear_ac_argmax_launch(static_cast<const b2e::f16*>(x), labels, (int)N, (int)Hi, (int)Wi, (int)P, (int)K, (int)S,
                                        (int)S, (cudaStream_t)stream, planes);
}
