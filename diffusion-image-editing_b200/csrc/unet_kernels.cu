// GroupNorm+SiLU, layout packing, upsampling, timestep embedding and attention kernels of the
// UNet.  All activations are f16 NHWC; statistics, softmax and accumulation are fp32/fp64.
#include "unet_kernels.cuh"
#include "gn_math.cuh"

#include <math.h>
#include <stdlib.h>

namespace b2e {

constexpr int kGNThreads = 256;

// ------------------------------------------------------------------ GroupNorm
// Thread layout: a "slot" is 8 consecutive channels (one 16-byte access); 256 / slots pixels are
// processed per sweep and four sweeps are unrolled so every thread keeps four independent 16-byte
// loads in flight.
constexpr int kGNUnroll = 4;

// (forward GroupNorm kernels: 256 threads, or 512 when the tensor has more than 2048 channels - SD concatenations)
template <bool SPLIT>
__global__ void __launch_bounds__(512) gn_partial_kernel(GNArgs a) {
  pdl_wait();
  __shared__ float s_sum[4096], s_sq[4096];
  const int C = a.C0 + a.C1, slots = C >> 3, ppi = (int)blockDim.x / slots;
  const int n = blockIdx.y, chunk = blockIdx.x, tid = threadIdx.x;
  const int s = tid % slots, pl = tid / slots;
  const int per = (a.HW + a.chunks - 1) / a.chunks;
  const int p0 = chunk * per, p1 = min(a.HW, p0 + per);
  if (pl < ppi) {
    float sum[8], sq[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) sum[j] = sq[j] = 0.f;
    const int c = s * 8;
    const f16* src; int cs, coff;
    if (c < a.C0) { src = a.x0; cs = a.P0; coff = c; } else { src = a.x1; cs = a.P1; coff = c - a.C0; }
    constexpr bool split = SPLIT;         // split-f16 tensors: value = plane 0 (hi) + plane 1 (lo), pixel pitch 3 * P
    const int lo_off = cs;
    cs *= a.planes;
    src += (int64_t)n * a.HW * cs + coff;
    for (int p = p0 + pl; p < p1; p += ppi * kGNUnroll) {
      uint4 v[kGNUnroll], w[kGNUnroll];
#pragma unroll
      for (int u = 0; u < kGNUnroll; ++u) {
        const int q = p + u * ppi;
        v[u] = q < p1 ? __ldg(reinterpret_cast<const uint4*>(src + (int64_t)q * cs)) : make_uint4(0, 0, 0, 0);
        w[u] = (split && q < p1) ? __ldg(reinterpret_cast<const uint4*>(src + (int64_t)q * cs + lo_off)) : make_uint4(0, 0, 0, 0);
      }
#pragma unroll
      for (int u = 0; u < kGNUnroll; ++u) {
        float f[8];
        unpack8(v[u], f);
        if (split) {
          float g[8];
          unpack8(w[u], g);
#pragma unroll
          for (int j = 0; j < 8; ++j) f[j] += g[j];
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) { sum[j] += f[j]; sq[j] += f[j] * f[j]; }
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) { s_sum[pl * C + c + j] = sum[j]; s_sq[pl * C + c + j] = sq[j]; }
  }
  __syncthreads();
  if (tid < a.G) {
    const int cpg = C / a.G;
    float ts = 0.f, tq = 0.f;
    for (int q = 0; q < ppi; ++q)
      for (int c = tid * cpg; c < (tid + 1) * cpg; ++c) { ts += s_sum[q * C + c]; tq += s_sq[q * C + c]; }
    float* o = a.partial + (((int64_t)n * a.chunks + chunk) * a.G + tid) * 2;
    o[0] = ts; o[1] = tq;
  }
}

template <bool SPLIT>
__global__ void __launch_bounds__(512, SPLIT ? 1 : 2) gn_apply_kernel(GNArgs a, int pix_per_block) {
  __shared__ float s_mean[64], s_rstd[64];
  extern __shared__ double s_ch[];          // [C][2]: per-channel (sum, sum of squares) of image n (fused-statistics paths)
  const int C = a.C0 + a.C1, slots = a.Pout >> 3, ppi = (int)blockDim.x / slots;
  // REVERSE block order (B2E_GN_REVERSE, default on): the producing convolution wrote the tensor front to back, so its
  // tail is what the 126 MB L2 still holds - start there; the normalised tensor is then written back to front and its
  // FRONT is what L2 holds when the consumer convolution starts at tile 0
  const int n = a.reverse ? (int)(gridDim.y - 1 - blockIdx.y) : (int)blockIdx.y, tid = threadIdx.x;
  const int bx = a.reverse ? (int)(gridDim.x - 1 - blockIdx.x) : (int)blockIdx.x;
  const int cpg = C / a.G;
  // role of this thread in the apply pass: 8 channels [c, c + 8) of every ppi-th pixel of the block's pixel range
  const int s = tid % slots, pl = tid / slots, c = s * 8;
  const int p0 = bx * pix_per_block, p1 = min(a.HW, p0 + pix_per_block);
  const bool streams = pl < ppi && c < C;
  const f16* src = nullptr; int cs = 0, lo_off = 0;
  if (streams) {
    int coff;
    if (c < a.C0) { src = a.x0; cs = a.P0; coff = c; } else { src = a.x1; cs = a.P1; coff = c - a.C0; }
    lo_off = cs;
    cs *= a.planes;
    src += (int64_t)n * a.HW * cs + coff;
  }
  // the affine parameters are weights (not written by the preceding kernel): fetch them before the grid dependency
  float scale[8], shift[8];
  if (streams) {
#pragma unroll
    for (int j = 0; j < 8; ++j) { scale[j] = __ldg(a.gamma + c + j); shift[j] = __ldg(a.beta + c + j); }
  }
  pdl_wait();
  // first sweep of the streaming pass: in flight while the statistics prologue below runs (plain tensors)
  uint4 v[kGNUnroll];
  if constexpr (!SPLIT) {
    if (streams) {
#pragma unroll
      for (int u = 0; u < kGNUnroll; ++u) {
        const int q = p0 + pl + u * ppi;
        if (q < p1) v[u] = __ldg(reinterpret_cast<const uint4*>(src + (int64_t)q * cs));
      }
    }
  }
  if (a.ts0 || a.cs0) {
    // statistics from the producing convolutions' epilogues (concat-aware): ALL threads gather the per-channel sums of
    // image n with independent loads in flight (one thread per group walking its channels serially exposed ~16-64
    // dependent L2 round trips: 10 of the 13 us of a low-resolution launch), then the group threads combine them
    for (int c = tid; c < C; c += blockDim.x) {
      const bool first = c < a.C0;
      const int Cs = first ? a.P0 : a.P1, cc = first ? c : c - a.C0;
      double ts = 0.0, tq = 0.0;
      if (a.ts0) {
        // raw tile statistics of a small tensor: slots of image n are (n/Nt * per_img + i) * Nt + n % Nt
        const float* t = first ? a.ts0 : a.ts1;
        const int64_t base = (int64_t)(n / a.ts_nt) * a.ts_per_img;
        const int nl = n % a.ts_nt;
#pragma unroll 4
        for (int i = 0; i < a.ts_per_img; ++i) {
          const float2 v = __ldg(reinterpret_cast<const float2*>(t + (((base + i) * a.ts_nt + nl) * Cs + cc) * 2));
          ts += (double)v.x; tq += (double)v.y;
        }
      } else {
        const float2 v = __ldg(reinterpret_cast<const float2*>((first ? a.cs0 : a.cs1) + ((int64_t)n * Cs + cc) * 2));
        ts = (double)v.x; tq = (double)v.y;
      }
      s_ch[2 * c] = ts; s_ch[2 * c + 1] = tq;
    }
    __syncthreads();
  }
  if (tid < a.G) {
    double ts = 0.0, tq = 0.0;
    if (a.ts0 || a.cs0) {
      for (int c = tid * cpg; c < (tid + 1) * cpg; ++c) { ts += s_ch[2 * c]; tq += s_ch[2 * c + 1]; }
    } else {
      for (int ch = 0; ch < a.chunks; ++ch) {
        const float* o = a.partial + (((int64_t)n * a.chunks + ch) * a.G + tid) * 2;
        ts += (double)o[0]; tq += (double)o[1];
      }
    }
    const double cnt = (double)a.HW * cpg;
    const double mean = ts / cnt;
    double var = tq / cnt - mean * mean;
    if (var < 0.0) var = 0.0;
    s_mean[tid] = (float)mean;
    s_rstd[tid] = (float)(1.0 / sqrt(var + (double)a.eps));
    if (a.save_stats && bx == 0)
      *reinterpret_cast<float2*>(a.save_stats + ((int64_t)n * a.G + tid) * 2) = make_float2(s_mean[tid], s_rstd[tid]);
  }
  __syncthreads();
  if (pl >= ppi) return;
  constexpr bool split = SPLIT;           // split-f16 tensors (fp32-accurate mode): planes [hi | lo | hi]
  const int po = a.Pout * a.planes;       // output pixel pitch
  f16* dst = a.out + (int64_t)n * a.HW * po + c;
  if (c >= C) {   // zero padding of the output pitch
    for (int p = p0 + pl; p < p1; p += ppi)
      for (int k = 0; k < a.planes; ++k) *reinterpret_cast<uint4*>(dst + (int64_t)p * po + k * a.Pout) = make_uint4(0, 0, 0, 0);
    return;
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int g = (c + j) / cpg;
    scale[j] = s_rstd[g] * scale[j];
    shift[j] = shift[j] - s_mean[g] * scale[j];
  }
  if constexpr (split) {
    // accurate path: x = hi + lo, exact-exp SiLU, output re-split into hi / lo (third plane repeats hi)
    for (int p = p0 + pl; p < p1; p += ppi * kGNUnroll) {
      uint4 v[kGNUnroll], w[kGNUnroll];
#pragma unroll
      for (int u = 0; u < kGNUnroll; ++u) {
        const int q = p + u * ppi;
        if (q < p1) {
          v[u] = __ldg(reinterpret_cast<const uint4*>(src + (int64_t)q * cs));
          w[u] = __ldg(reinterpret_cast<const uint4*>(src + (int64_t)q * cs + lo_off));
        }
      }
#pragma unroll
      for (int u = 0; u < kGNUnroll; ++u) {
        const int q = p + u * ppi;
        if (q < p1) {
          float f[8], g[8], l[8];
          unpack8(v[u], f);
          unpack8(w[u], g);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float y = fmaf(f[j] + g[j], scale[j], shift[j]);
            if (a.silu) y = y / (1.f + expf(-y));
            f[j] = y;
            l[j] = __fsub_rn(y, f16_to_float(float_to_f16(y)));
          }
          const uint4 hi = pack8(f), lo = pack8(l);
          f16* o = dst + (int64_t)q * po;
          *reinterpret_cast<uint4*>(o) = hi;
          *reinterpret_cast<uint4*>(o + a.Pout) = lo;
          *reinterpret_cast<uint4*>(o + 2 * a.Pout) = hi;
        }
      }
    }
    return;
  }
  // double-buffered sweeps: the loads of sweep i + 1 are issued before sweep i is transformed and stored
  for (int p = p0 + pl; p < p1; p += ppi * kGNUnroll) {
    uint4 w[kGNUnroll];
    const int pn = p + ppi * kGNUnroll;
#pragma unroll
    for (int u = 0; u < kGNUnroll; ++u) {
      const int q = pn + u * ppi;
      if (q < p1) w[u] = __ldg(reinterpret_cast<const uint4*>(src + (int64_t)q * cs));
    }
#pragma unroll
    for (int u = 0; u < kGNUnroll; ++u) {
      const int q = p + u * ppi;
      if (q < p1) *reinterpret_cast<uint4*>(dst + (int64_t)q * a.Pout) = gn_apply8(v[u], scale, shift, a.silu != 0);
    }
#pragma unroll
    for (int u = 0; u < kGNUnroll; ++u) v[u] = w[u];
  }
}

// Bulk-copy variant of the apply pass (plain f16 tensors - channel pitches allowed -, statistics from the producing
// convolution): thread 0 issues the block's whole input - one contiguous chunk per source - as cp.async.bulk copies into
// shared memory BEFORE the statistics prologue, so up to 64 KB per block are in flight while the prologue runs, without
// holding them in registers; the transform then reads shared memory.  Same arithmetic, same results as gn_apply_kernel.
__global__ void __launch_bounds__(kGNThreads) gn_apply_bulk_kernel(GNArgs a, int pix_per_block) {
  __shared__ float s_mean[64], s_rstd[64];
  __shared__ __align__(8) uint64_t s_bar;
  extern __shared__ __align__(128) uint8_t s_dyn[];
  const int C = a.C0 + a.C1, slots = a.Pout >> 3, ppi = (int)blockDim.x / slots;
  const int n = a.reverse ? (int)(gridDim.y - 1 - blockIdx.y) : (int)blockIdx.y, tid = threadIdx.x;
  const int bx = a.reverse ? (int)(gridDim.x - 1 - blockIdx.x) : (int)blockIdx.x;
  const int cpg = C / a.G;
  const int p0 = bx * pix_per_block, p1 = min(a.HW, p0 + pix_per_block), np = p1 - p0;
  // [x0 chunk: np x P0][x1 chunk: np x P1] f16 (channel pitches as in memory), then the per-channel sums (doubles)
  f16* t0 = reinterpret_cast<f16*>(s_dyn);
  f16* t1 = t0 + (size_t)pix_per_block * a.P0;
  double* s_ch = reinterpret_cast<double*>(s_dyn + (size_t)pix_per_block * (a.P0 + a.P1) * sizeof(f16));
  const int s = tid % slots, pl = tid / slots, c = s * 8;
  const bool live = c < C;     // slots beyond the real channels write the zero padding of the output pitch
  float scale[8], shift[8];
  if (live) {
#pragma unroll
    for (int j = 0; j < 8; ++j) { scale[j] = __ldg(a.gamma + c + j); shift[j] = __ldg(a.beta + c + j); }
  }
  const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&s_bar);
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  pdl_wait();
  if (tid == 0) {
    const uint32_t b0 = (uint32_t)np * a.P0 * sizeof(f16), b1 = a.C1 ? (uint32_t)np * a.P1 * sizeof(f16) : 0u;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(b0 + b1) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"((uint32_t)__cvta_generic_to_shared(t0)), "l"(a.x0 + ((int64_t)n * a.HW + p0) * a.P0), "r"(b0), "r"(bar) : "memory");
    if (b1)
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"((uint32_t)__cvta_generic_to_shared(t1)), "l"(a.x1 + ((int64_t)n * a.HW + p0) * a.P1), "r"(b1), "r"(bar) : "memory");
  }
  // statistics prologue (as gn_apply_kernel)
  for (int ch = tid; ch < C; ch += blockDim.x) {
    const bool first = ch < a.C0;
    const int Cs = first ? a.P0 : a.P1, cc = first ? ch : ch - a.C0;
    double ts = 0.0, tq = 0.0;
    if (a.ts0) {
      const float* t = first ? a.ts0 : a.ts1;
      const int64_t base = (int64_t)(n / a.ts_nt) * a.ts_per_img;
      const int nl = n % a.ts_nt;
#pragma unroll 4
      for (int i = 0; i < a.ts_per_img; ++i) {
        const float2 v = __ldg(reinterpret_cast<const float2*>(t + (((base + i) * a.ts_nt + nl) * Cs + cc) * 2));
        ts += (double)v.x; tq += (double)v.y;
      }
    } else {
      const float2 v = __ldg(reinterpret_cast<const float2*>((first ? a.cs0 : a.cs1) + ((int64_t)n * Cs + cc) * 2));
      ts = (double)v.x; tq = (double)v.y;
    }
    s_ch[2 * ch] = ts; s_ch[2 * ch + 1] = tq;
  }
  __syncthreads();
  if (tid < a.G) {
    double ts = 0.0, tq = 0.0;
    for (int ch = tid * cpg; ch < (tid + 1) * cpg; ++ch) { ts += s_ch[2 * ch]; tq += s_ch[2 * ch + 1]; }
    const double cnt = (double)a.HW * cpg;
    const double mean = ts / cnt;
    double var = tq / cnt - mean * mean;
    if (var < 0.0) var = 0.0;
    s_mean[tid] = (float)mean;
    s_rstd[tid] = (float)(1.0 / sqrt(var + (double)a.eps));
    if (a.save_stats && bx == 0)
      *reinterpret_cast<float2*>(a.save_stats + ((int64_t)n * a.G + tid) * 2) = make_float2(s_mean[tid], s_rstd[tid]);
  }
  __syncthreads();
  if (pl >= ppi) return;
  f16* dst = a.out + ((int64_t)n * a.HW + p0) * a.Pout + c;
  if (!live) {
    for (int q = pl; q < np; q += ppi) *reinterpret_cast<uint4*>(dst + (int64_t)q * a.Pout) = make_uint4(0, 0, 0, 0);
    return;
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int g = (c + j) / cpg;
    scale[j] = s_rstd[g] * scale[j];
    shift[j] = shift[j] - s_mean[g] * scale[j];
  }
  // wait for the chunk(s)
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "GNB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], 0;\n"
      "@P1 bra GNB_DONE;\n"
      "bra GNB_WAIT;\n"
      "GNB_DONE:\n"
      "}\n" ::"r"(bar) : "memory");
  const bool first = c < a.C0;
  const f16* src = first ? t0 + c : t1 + (c - a.C0);
  const int cs = first ? a.P0 : a.P1;
#pragma unroll 4
  for (int q = pl; q < np; q += ppi) {
    const uint4 v = *reinterpret_cast<const uint4*>(src + (size_t)q * cs);
    *reinterpret_cast<uint4*>(dst + (int64_t)q * a.Pout) = gn_apply8(v, scale, shift, a.silu != 0);
  }
}

// Coefficients of the FUSED GroupNorm (conv_igemm XF kernels): per image n and per K position p of the consumer
// convolution's A operand (source 0 at [0, P0), source 1 at [P0, P0 + P1), pitches included) the pair
// (scale, shift) = (rstd_g gamma_c, beta_c - mean_g scale) - the arithmetic of gn_apply_kernel - and (0, 0) on the zero
// tails of pitched sources.  One block per image; statistics from the producing convolutions' epilogues (per-channel
// sums cs*, or raw tile slots ts* of small tensors) or from the stand-alone gn_partial pass.
__global__ void __launch_bounds__(256) gn_coeffs_kernel(GNArgs a, float2* __restrict__ coef) {
  pdl_wait();
  pdl_trigger();
  extern __shared__ double s_ch[];          // [C][2] per-channel (sum, sum of squares) of image n
  __shared__ float s_mean[64], s_rstd[64];
  const int C = a.C0 + a.C1, n = blockIdx.x, tid = threadIdx.x;
  const int cpg = C / a.G;
  if (a.ts0 || a.cs0) {
    for (int c = tid; c < C; c += blockDim.x) {
      const bool first = c < a.C0;
      const int Cs = first ? a.P0 : a.P1, cc = first ? c : c - a.C0;
      double ts = 0.0, tq = 0.0;
      if (a.ts0) {
        const float* t = first ? a.ts0 : a.ts1;
        const int64_t base = (int64_t)(n / a.ts_nt) * a.ts_per_img;
        const int nl = n % a.ts_nt;
        for (int i = 0; i < a.ts_per_img; ++i) {
          const float2 v = __ldg(reinterpret_cast<const float2*>(t + (((base + i) * a.ts_nt + nl) * Cs + cc) * 2));
          ts += (double)v.x; tq += (double)v.y;
        }
      } else {
        const float* o = (first ? a.cs0 : a.cs1) + ((int64_t)n * Cs + cc) * 2;
        ts = (double)o[0]; tq = (double)o[1];
      }
      s_ch[2 * c] = ts; s_ch[2 * c + 1] = tq;
    }
    __syncthreads();
  }
  if (tid < a.G) {
    double ts = 0.0, tq = 0.0;
    if (a.ts0 || a.cs0) {
      for (int c = tid * cpg; c < (tid + 1) * cpg; ++c) { ts += s_ch[2 * c]; tq += s_ch[2 * c + 1]; }
    } else {
      for (int ch = 0; ch < a.chunks; ++ch) {
        const float* o = a.partial + (((int64_t)n * a.chunks + ch) * a.G + tid) * 2;
        ts += (double)o[0]; tq += (double)o[1];
      }
    }
    const double cnt = (double)a.HW * cpg;
    const double mean = ts / cnt;
    double var = tq / cnt - mean * mean;
    if (var < 0.0) var = 0.0;
    s_mean[tid] = (float)mean;
    s_rstd[tid] = (float)(1.0 / sqrt(var + (double)a.eps));
    if (a.save_stats) *reinterpret_cast<float2*>(a.save_stats + ((int64_t)n * a.G + tid) * 2) = make_float2(s_mean[tid], s_rstd[tid]);
  }
  __syncthreads();
  const int K = a.P0 + a.P1;
  for (int p = tid; p < K; p += blockDim.x) {
    const bool first = p < a.P0;
    const int q = first ? p : p - a.P0;
    float2 o = make_float2(0.f, 0.f);
    if (q < (first ? a.C0 : a.C1)) {
      const int c = first ? q : a.C0 + q;
      const int g = c / cpg;
      o.x = s_rstd[g] * __ldg(a.gamma + c);
      o.y = __ldg(a.beta + c) - s_mean[g] * o.x;
    }
    coef[(int64_t)n * K + p] = o;
  }
}

int gn_coeffs_launch(const GNArgs& a, float* coef, cudaStream_t st) {
  const int C = a.C0 + a.C1;
  B2E_REQUIRE(C % 8 == 0 && a.C0 % 8 == 0 && a.G <= 64 && C % a.G == 0 && a.planes == 1, B2E_UNSUPPORTED_SHAPE,
              "groupnorm coefficients: unsupported channels %d+%d / groups %d", a.C0, a.C1, a.G);
  int rc = B2E_OK;
  if (!a.cs0 && !a.ts0) {   // no statistics from a producing convolution: stand-alone pass over the raw tensor(s)
    launch_pdl(gn_partial_kernel<false>, dim3(dim3(a.chunks, a.N)), dim3(C > 2048 ? 512 : kGNThreads), 0, st, a);
    rc = check_launch("gn_partial");
    if (rc) return rc;
  }
  const size_t smem = sizeof(double) * 2 * (size_t)C;
  static bool attr_set = false;
  if (!attr_set) {
    B2E_CUDA(cudaFuncSetAttribute(gn_coeffs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    attr_set = true;
  }
  B2E_REQUIRE(smem <= 96 * 1024, B2E_UNSUPPORTED_SHAPE, "groupnorm coefficients: %d channels", C);
  launch_pdl(gn_coeffs_kernel, dim3(a.N), dim3(256), smem, st, a, reinterpret_cast<float2*>(coef));
  return check_launch("gn_coeffs");
}

int gn_chunks(int HW, int C) {
  // ~16K elements (two unrolled sweeps) per block, at most 64 partial rows per image
  int64_t el = (int64_t)HW * C;
  int ch = (int)((el + 16383) / 16384);
  if (ch < 1) ch = 1;
  if (ch > 64) ch = 64;
  return ch;
}

int gn_launch(const GNArgs& a_in, cudaStream_t st) {
  static const int rev = getenv("B2E_GN_REVERSE") ? atoi(getenv("B2E_GN_REVERSE")) : 1;
  GNArgs a = a_in;
  a.reverse = rev;
  const int C = a.C0 + a.C1;
  B2E_REQUIRE(C % 8 == 0 && a.C0 % 8 == 0 && a.Pout <= 4096 && a.G <= 64 && C % a.G == 0, B2E_UNSUPPORTED_SHAPE,
              "groupnorm: unsupported channels %d+%d / groups %d", a.C0, a.C1, a.G);
  B2E_REQUIRE(a.P0 >= a.C0 && a.P1 >= a.C1 && a.Pout >= C && a.P0 % 8 == 0 && a.P1 % 8 == 0 && a.Pout % 8 == 0,
              B2E_INVALID_ARG, "groupnorm: bad channel pitches %d/%d -> %d", a.P0, a.P1, a.Pout);
  B2E_REQUIRE(a.planes == 1 || (a.planes == 3 && !a.cs0 && !a.ts0 && !a.save_stats), B2E_INVALID_ARG,
              "groupnorm: split-f16 tensors take their statistics from the stand-alone pass");
  int rc = B2E_OK;
  if (!a.cs0 && !a.ts0) {
    if (a.planes == 3) launch_pdl(gn_partial_kernel<true>, dim3(dim3(a.chunks, a.N)), dim3(C > 2048 ? 512 : kGNThreads), 0, st, a);
    else launch_pdl(gn_partial_kernel<false>, dim3(dim3(a.chunks, a.N)), dim3(C > 2048 ? 512 : kGNThreads), 0, st, a);
    rc = check_launch("gn_partial");
    if (rc) return rc;
  }
  const int threads = a.Pout > 2048 ? 512 : kGNThreads;
  const int slots = a.Pout / 8, ppi = threads / slots;
  int ppb = ppi * kGNUnroll * 2;  // two unrolled sweeps per thread
  if (ppb > a.HW) ppb = a.HW;
  const size_t smem = (a.cs0 || a.ts0) ? sizeof(double) * 2 * (size_t)C : 0;   // per-channel sums of the fused-statistics paths
  static bool attr_set = false;
  if (!attr_set) {
    B2E_CUDA(cudaFuncSetAttribute(gn_apply_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    attr_set = true;
  }
  // bulk-copy variant: plain tensors with compact channels and fused statistics.  Chunk per block (measured on B200 at batch 8,
  // all GroupNorm launches of a DDPM-256 forward, tools/profile_ops.py: stand-alone kernel 1.573 ms; 8 / 16 / 32 / 48 / 64 / 96 /
  // 128 KB chunks 2.89 / 1.94 / 1.515 / 1.459 / 1.449 / 1.51 / 1.70 ms): 64 KB where that still gives two waves of blocks
  // (the 256x256 concatenated layers: 104 -> 86 us = 0.93 of the HBM copy peak), 32 KB for mid-size tensors of <= 256
  // channels, the register-staged kernel below for everything smaller.  B2E_GN_BULK=0 disables, B2E_GN_BULK_KB forces a size.
  static const int bulk_on = getenv("B2E_GN_BULK") ? atoi(getenv("B2E_GN_BULK")) : 1;
  static const int bulk_kb = getenv("B2E_GN_BULK_KB") ? atoi(getenv("B2E_GN_BULK_KB")) : 0;
  const int64_t tensor_bytes = (int64_t)a.N * a.HW * C * 2;
  int bulk_bytes = bulk_kb > 0 ? bulk_kb * 1024
                               : tensor_bytes >= (int64_t)2 * kNumSMs * 65536 ? 65536
                               : (tensor_bytes >= (int64_t)8 << 20 && C <= 256) ? 32768 : 0;
  const int Pin = a.P0 + (a.C1 ? a.P1 : 0);     // input f16 per pixel as stored (channel pitches: LDM's 224 -> 256, ...)
  if (bulk_on && bulk_bytes && a.planes == 1 && (a.cs0 || a.ts0) && Pin <= 2048 && threads == kGNThreads &&
      (int64_t)a.HW * Pin * 2 >= 2 * (int64_t)bulk_bytes) {
    int bp = bulk_bytes / (Pin * 2);           // pixels per block: a multiple of the pixel lanes
    bp -= bp % ppi;
    if (bp >= ppi) {
      const size_t bsmem = (size_t)bp * Pin * sizeof(f16) + sizeof(double) * 2 * (size_t)C;
      static bool battr = false;
      if (!battr) {
        B2E_CUDA(cudaFuncSetAttribute(gn_apply_bulk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        battr = true;
      }
      launch_pdl(gn_apply_bulk_kernel, dim3(dim3((a.HW + bp - 1) / bp, a.N)), dim3(threads), bsmem, st, a, bp);
      return check_launch("gn_apply_bulk");
    }
  }
  if (a.planes == 3) launch_pdl(gn_apply_kernel<true>, dim3(dim3((a.HW + ppb - 1) / ppb, a.N)), dim3(threads), smem, st, a, ppb);
  else launch_pdl(gn_apply_kernel<false>, dim3(dim3((a.HW + ppb - 1) / ppb, a.N)), dim3(threads), smem, st, a, ppb);
  return check_launch("gn_apply");
}

// ------------------------------------------------------------------ GroupNorm (+SiLU) backward
// silu'(y) = s (1 + y (1 - s)), s = sigmoid(y) = 0.5 + 0.5 tanh(y / 2): one MUFU op
__device__ __forceinline__ float silu_grad(float y) {
  float th;
  asm("tanh.approx.f32 %0, %1;" : "=f"(th) : "f"(0.5f * y));
  const float sg = fmaf(0.5f, th, 0.5f);
  return sg * fmaf(y, 1.f - sg, 1.f);
}

// Per-channel constants of the backward pass: y = x*sc + sh (the forward's affine), xh = x*r + mr (normalised input).
// Both kernels keep several independent 16-byte loads in flight per thread (the loops are latency-bound otherwise:
// measured 1.6 TB/s before unrolling against 5 TB/s for the forward apply kernel).
constexpr int kGNBwdUnroll = 4;   // measured at batch 32 (decoder backward, 24 launches): unroll 2 16.9 ms, 4 13.0 ms, 8 15.4 ms

__global__ void __launch_bounds__(kGNThreads) gn_bwd_partial_kernel(GNBwdArgs a) {
  pdl_wait();
  __shared__ float s_a[2048], s_b[2048];
  const int C = a.C, slots = C >> 3, ppi = kGNThreads / slots;
  const int n = blockIdx.y, chunk = blockIdx.x, tid = threadIdx.x;
  const int s = tid % slots, pl = tid / slots;
  const int per = (a.HW + a.chunks - 1) / a.chunks;
  const int p0 = chunk * per, p1 = min(a.HW, p0 + per);
  const int cpg = C / a.G;
  if (pl < ppi) {
    float sa[8], sb[8], sc[8], sh[8], r[8], mr[8], gam[8];
    const int c = s * 8;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      sa[j] = sb[j] = 0.f;
      const float2 st = *reinterpret_cast<const float2*>(a.stats + ((int64_t)n * a.G + (c + j) / cpg) * 2);
      gam[j] = __ldg(a.gamma + c + j);
      r[j] = st.y; mr[j] = -st.x * st.y;
      sc[j] = gam[j] * st.y; sh[j] = fmaf(gam[j], mr[j], __ldg(a.beta + c + j));
    }
    const f16* xs = a.x + (int64_t)n * a.HW * a.P + c;
    const f16* ds = a.da + (int64_t)n * a.HW * a.Pda + c;
    for (int p = p0 + pl; p < p1; p += ppi * kGNBwdUnroll) {
      uint4 xv[kGNBwdUnroll], dv[kGNBwdUnroll];
#pragma unroll
      for (int u = 0; u < kGNBwdUnroll; ++u) {
        const int q = p + u * ppi;
        if (q < p1) {
          xv[u] = __ldg(reinterpret_cast<const uint4*>(xs + (int64_t)q * a.P));
          dv[u] = __ldg(reinterpret_cast<const uint4*>(ds + (int64_t)q * a.Pda));
        }
      }
#pragma unroll
      for (int u = 0; u < kGNBwdUnroll; ++u) {
        if (p + u * ppi < p1) {
          float xf[8], df[8];
          unpack8(xv[u], xf);
          unpack8(dv[u], df);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float dy = df[j];
            if (a.silu) dy *= silu_grad(fmaf(xf[j], sc[j], sh[j]));
            const float dxh = dy * gam[j];
            sa[j] += dxh; sb[j] = fmaf(dxh, fmaf(xf[j], r[j], mr[j]), sb[j]);
          }
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) { s_a[pl * C + c + j] = sa[j]; s_b[pl * C + c + j] = sb[j]; }
  }
  __syncthreads();
  if (tid < a.G) {
    float ta = 0.f, tb = 0.f;
    for (int q = 0; q < ppi; ++q)
      for (int c = tid * cpg; c < (tid + 1) * cpg; ++c) { ta += s_a[q * C + c]; tb += s_b[q * C + c]; }
    float* o = a.partial + (((int64_t)n * a.chunks + chunk) * a.G + tid) * 2;
    o[0] = ta; o[1] = tb;
  }
}

__global__ void __launch_bounds__(kGNThreads) gn_bwd_apply_kernel(GNBwdArgs a, int pix_per_block) {
  pdl_wait();
  __shared__ float s_ma[64], s_mb[64];
  const int C = a.C, slots = a.P >> 3, ppi = kGNThreads / slots;
  const int n = blockIdx.y, tid = threadIdx.x;
  const int cpg = C / a.G;
  if (tid < a.G) {
    double ta = 0.0, tb = 0.0;
    for (int ch = 0; ch < a.chunks; ++ch) {
      const float* o = a.partial + (((int64_t)n * a.chunks + ch) * a.G + tid) * 2;
      ta += (double)o[0]; tb += (double)o[1];
    }
    const double cnt = (double)a.HW * cpg;
    s_ma[tid] = (float)(ta / cnt); s_mb[tid] = (float)(tb / cnt);
  }
  __syncthreads();
  const int s = tid % slots, pl = tid / slots;
  if (pl >= ppi) return;
  const int c = s * 8;
  const int p0 = blockIdx.x * pix_per_block, p1 = min(a.HW, p0 + pix_per_block);
  f16* dst = a.dx + (int64_t)n * a.HW * a.P + c;
  if (c >= C) {
    for (int p = p0 + pl; p < p1; p += ppi) *reinterpret_cast<uint4*>(dst + (int64_t)p * a.P) = make_uint4(0, 0, 0, 0);
    return;
  }
  // dx = rstd * (dy*gam - ma - xh*mb) = dy * gr + x * k1 + k0 with gr = gam*rstd, k1 = -rstd*r*mb, k0 = -rstd*(ma + mr*mb)
  float sc[8], sh[8], gr[8], k1[8], k0[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int g = (c + j) / cpg;
    const float2 st = *reinterpret_cast<const float2*>(a.stats + ((int64_t)n * a.G + g) * 2);
    const float gam = __ldg(a.gamma + c + j), rstd = st.y, mr = -st.x * st.y;
    sc[j] = gam * rstd; sh[j] = fmaf(gam, mr, __ldg(a.beta + c + j));
    gr[j] = gam * rstd;
    k1[j] = -rstd * rstd * s_mb[g];
    k0[j] = -rstd * fmaf(mr, s_mb[g], s_ma[g]);
  }
  const f16* xs = a.x + (int64_t)n * a.HW * a.P + c;
  const f16* ds = a.da + (int64_t)n * a.HW * a.Pda + c;
  const f16* as = a.add ? a.add + (int64_t)n * a.HW * a.P + c : nullptr;
  for (int p = p0 + pl; p < p1; p += ppi * kGNBwdUnroll) {
    uint4 xv[kGNBwdUnroll], dv[kGNBwdUnroll], av[kGNBwdUnroll];
#pragma unroll
    for (int u = 0; u < kGNBwdUnroll; ++u) {
      const int q = p + u * ppi;
      if (q < p1) {
        xv[u] = __ldg(reinterpret_cast<const uint4*>(xs + (int64_t)q * a.P));
        dv[u] = __ldg(reinterpret_cast<const uint4*>(ds + (int64_t)q * a.Pda));
        if (as) av[u] = __ldg(reinterpret_cast<const uint4*>(as + (int64_t)q * a.P));
      }
    }
#pragma unroll
    for (int u = 0; u < kGNBwdUnroll; ++u) {
      const int q = p + u * ppi;
      if (q < p1) {
        float xf[8], df[8], af[8];
        unpack8(xv[u], xf);
        unpack8(dv[u], df);
        if (as) unpack8(av[u], af);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float dy = df[j];
          if (a.silu) dy *= silu_grad(fmaf(xf[j], sc[j], sh[j]));
          float dx = fmaf(dy, gr[j], fmaf(xf[j], k1[j], k0[j]));
          if (as) dx += af[j];
          xf[j] = dx;
        }
        *reinterpret_cast<uint4*>(dst + (int64_t)q * a.P) = pack8(xf);
      }
    }
  }
}

// Bulk-copy variant of the backward apply pass (compact channels: C == P == Pda): the block's x / da / add chunks are issued
// as cp.async.bulk copies into shared memory before the per-group prologue (see gn_apply_bulk_kernel).  Same arithmetic.
__global__ void __launch_bounds__(kGNThreads) gn_bwd_apply_bulk_kernel(GNBwdArgs a, int pix_per_block) {
  __shared__ float s_ma[64], s_mb[64];
  __shared__ __align__(8) uint64_t s_bar;
  extern __shared__ __align__(128) uint8_t s_dyn[];
  const int C = a.C, slots = C >> 3, ppi = kGNThreads / slots;
  const int n = blockIdx.y, tid = threadIdx.x;
  const int cpg = C / a.G;
  const int p0 = blockIdx.x * pix_per_block, p1 = min(a.HW, p0 + pix_per_block), np = p1 - p0;
  f16* tx = reinterpret_cast<f16*>(s_dyn);
  f16* td = tx + (size_t)pix_per_block * C;
  f16* ta = td + (size_t)pix_per_block * C;
  const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&s_bar);
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  pdl_wait();
  if (tid == 0) {
    const uint32_t bytes = (uint32_t)np * C * sizeof(f16);
    const int64_t off = ((int64_t)n * a.HW + p0) * C;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes * (a.add ? 3u : 2u)) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"((uint32_t)__cvta_generic_to_shared(tx)), "l"(a.x + off), "r"(bytes), "r"(bar) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"((uint32_t)__cvta_generic_to_shared(td)), "l"(a.da + off), "r"(bytes), "r"(bar) : "memory");
    if (a.add)
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"((uint32_t)__cvta_generic_to_shared(ta)), "l"(a.add + off), "r"(bytes), "r"(bar) : "memory");
  }
  if (tid < a.G) {
    double ta2 = 0.0, tb2 = 0.0;
    for (int ch = 0; ch < a.chunks; ++ch) {
      const float* o = a.partial + (((int64_t)n * a.chunks + ch) * a.G + tid) * 2;
      ta2 += (double)o[0]; tb2 += (double)o[1];
    }
    const double cnt = (double)a.HW * cpg;
    s_ma[tid] = (float)(ta2 / cnt); s_mb[tid] = (float)(tb2 / cnt);
  }
  __syncthreads();
  const int s = tid % slots, pl = tid / slots;
  if (pl >= ppi) return;
  const int c = s * 8;
  float sc[8], sh[8], gr[8], k1[8], k0[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int g = (c + j) / cpg;
    const float2 st = *reinterpret_cast<const float2*>(a.stats + ((int64_t)n * a.G + g) * 2);
    const float gam = __ldg(a.gamma + c + j), rstd = st.y, mr = -st.x * st.y;
    sc[j] = gam * rstd; sh[j] = fmaf(gam, mr, __ldg(a.beta + c + j));
    gr[j] = gam * rstd;
    k1[j] = -rstd * rstd * s_mb[g];
    k0[j] = -rstd * fmaf(mr, s_mb[g], s_ma[g]);
  }
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "GNBB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], 0;\n"
      "@P1 bra GNBB_DONE;\n"
      "bra GNBB_WAIT;\n"
      "GNBB_DONE:\n"
      "}\n" ::"r"(bar) : "memory");
  f16* dst = a.dx + ((int64_t)n * a.HW + p0) * C + c;
  const bool has_add = a.add != nullptr;
#pragma unroll 2
  for (int q = pl; q < np; q += ppi) {
    float xf[8], df[8], af[8];
    unpack8(*reinterpret_cast<const uint4*>(tx + (size_t)q * C + c), xf);
    unpack8(*reinterpret_cast<const uint4*>(td + (size_t)q * C + c), df);
    if (has_add) unpack8(*reinterpret_cast<const uint4*>(ta + (size_t)q * C + c), af);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float dy = df[j];
      if (a.silu) dy *= silu_grad(fmaf(xf[j], sc[j], sh[j]));
      float dx = fmaf(dy, gr[j], fmaf(xf[j], k1[j], k0[j]));
      if (has_add) dx += af[j];
      xf[j] = dx;
    }
    *reinterpret_cast<uint4*>(dst + (int64_t)q * C) = pack8(xf);
  }
}

int gn_bwd_launch(const GNBwdArgs& a, cudaStream_t st) {
  B2E_REQUIRE(a.C % 8 == 0 && a.P >= a.C && a.Pda >= a.C && a.P % 8 == 0 && a.Pda % 8 == 0 && a.P <= 2048 && a.G <= 64 &&
                  a.C % a.G == 0 && a.x && a.da && a.dx && a.stats && a.partial,
              B2E_UNSUPPORTED_SHAPE, "groupnorm backward: unsupported channels %d (pitch %d) / groups %d", a.C, a.P, a.G);
  const int slots = a.P / 8, ppi = kGNThreads / slots;
  int ppb = ppi * kGNBwdUnroll * 2;   // two unrolled sweeps per thread
  if (ppb > a.HW) ppb = a.HW;
  // Optional L2 blocking (B2E_GN_L2_MB = operand megabytes per group of images; default 0 = the whole batch in one pair of
  // launches): running the two passes back to back per group would turn the apply pass's re-read of x / da into L2 hits.
  // Measured at batch 32 (decoder backward, r90): 12.5 ms unblocked, 17.2 / 21.1 / 22.6 ms with 96 / 64 / 32 MB groups -
  // the statistics pass of a 2-3 image group (<= 192 blocks) no longer fills the chip - so it stays off.
  static const int l2_mb = getenv("B2E_GN_L2_MB") ? atoi(getenv("B2E_GN_L2_MB")) : 0;
  const int64_t per_img = (int64_t)a.HW * (a.P + a.Pda + (a.add ? a.P : 0)) * (int64_t)sizeof(f16);
  int group = a.N;
  if (l2_mb > 0 && per_img * a.N > (int64_t)l2_mb << 20) {
    group = (int)(((int64_t)l2_mb << 20) / per_img);
    if (group < 1) group = 1;
  }
  for (int n0 = 0; n0 < a.N; n0 += group) {
    GNBwdArgs g = a;
    g.N = a.N - n0 < group ? a.N - n0 : group;
    g.x = a.x + (int64_t)n0 * a.HW * a.P;
    g.da = a.da + (int64_t)n0 * a.HW * a.Pda;
    g.add = a.add ? a.add + (int64_t)n0 * a.HW * a.P : nullptr;
    g.dx = a.dx + (int64_t)n0 * a.HW * a.P;
    g.stats = a.stats + (int64_t)n0 * a.G * 2;
    g.partial = a.partial + (int64_t)n0 * a.chunks * a.G * 2;
    launch_pdl(gn_bwd_partial_kernel, dim3(g.chunks, g.N), dim3(kGNThreads), 0, st, g);
    int rc = check_launch("gn_bwd_partial");
    if (rc) return rc;
    // bulk-copy variant (compact channels): 64 KB of inputs per block where the grid keeps two waves, else 32 KB
    static const int bulk_on = getenv("B2E_GN_BULK") ? atoi(getenv("B2E_GN_BULK")) : 1;
    const int streams = g.add ? 3 : 2;
    const int64_t in_bytes = (int64_t)g.N * g.HW * g.C * 2 * streams;
    const int bulk_bytes = in_bytes >= (int64_t)2 * kNumSMs * 65536 ? 65536 : in_bytes >= (int64_t)8 << 20 ? 32768 : 0;
    int bp = bulk_bytes ? bulk_bytes / (g.C * 2 * streams) : 0;
    if (bp) bp -= bp % ppi;
    if (bulk_on && bp >= ppi && g.C == g.P && g.C == g.Pda && g.C <= 1024) {
      static bool battr = false;
      if (!battr) {
        B2E_CUDA(cudaFuncSetAttribute(gn_bwd_apply_bulk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        battr = true;
      }
      launch_pdl(gn_bwd_apply_bulk_kernel, dim3((g.HW + bp - 1) / bp, g.N), dim3(kGNThreads), (size_t)bp * g.C * 2 * streams, st, g, bp);
      rc = check_launch("gn_bwd_apply_bulk");
      if (rc) return rc;
      continue;
    }
    launch_pdl(gn_bwd_apply_kernel, dim3((g.HW + ppb - 1) / ppb, g.N), dim3(kGNThreads), 0, st, g, ppb);
    rc = check_launch("gn_bwd_apply");
    if (rc) return rc;
  }
  return B2E_OK;
}

// block = 16 channels x L slot lanes (L = 16, or 64 for images of >= 256 tile slots: a 256x256 layer has 512, and 16
// lanes walked them in four dependent rounds of loads - 11 us at batch 1): every thread sums a strided subset of the
// image's tile slots (independent loads in flight), then the lanes are combined in a fixed order through smem.
template <int L>
__global__ void __launch_bounds__(16 * L)
gn_finalize_kernel(const float* __restrict__ tile_stats, float* __restrict__ chan_stats, int C, int Nt, int w_blks,
                   int h_blks, int phases, int64_t phase_stride) {
  pdl_wait();
  pdl_trigger();
  __shared__ double s_s[L][16], s_q[L][16];
  const int cl = threadIdx.x & 15, sl = threadIdx.x >> 4;
  const int c = blockIdx.x * 16 + cl, n = blockIdx.y;
  const int n_blk = n / Nt, nl = n % Nt;
  const int per_img = h_blks * w_blks;
  double s = 0.0, q = 0.0;
  if (c < C) {
    const int64_t base = (int64_t)n_blk * per_img;
#pragma unroll 8
    // phases > 1: the tensor was written by `phases` launches (sub-pixel phases of an upsampling convolution), each with
    // its own block of slots `phase_stride` floats apart
    for (int i = sl; i < per_img * phases; i += L) {
      const int ph = i / per_img, ii = i - ph * per_img;
      const int64_t slot = (base + ii) * Nt + nl;
      const float2 v = __ldg(reinterpret_cast<const float2*>(tile_stats + ph * phase_stride + (slot * C + c) * 2));
      s += (double)v.x; q += (double)v.y;
    }
  }
  s_s[sl][cl] = s; s_q[sl][cl] = q;
  __syncthreads();
  if (sl == 0 && c < C) {
    double ts = 0.0, tq = 0.0;
#pragma unroll
    for (int i = 0; i < L; ++i) { ts += s_s[i][cl]; tq += s_q[i][cl]; }
    *reinterpret_cast<float2*>(chan_stats + ((int64_t)n * C + c) * 2) = make_float2((float)ts, (float)tq);
  }
}

int gn_finalize_launch(const float* tile_stats, float* chan_stats, int N, int C, int Nt, int w_blks, int h_blks,
                       cudaStream_t st, int phases, int64_t phase_stride) {
  if (w_blks * h_blks * phases >= 256)
    launch_pdl(gn_finalize_kernel<64>, dim3(dim3((C + 15) / 16, N)), dim3(1024), 0, st, tile_stats, chan_stats, C, Nt, w_blks, h_blks,
               phases, phase_stride);
  else
    launch_pdl(gn_finalize_kernel<16>, dim3(dim3((C + 15) / 16, N)), dim3(256), 0, st, tile_stats, chan_stats, C, Nt, w_blks, h_blks,
               phases, phase_stride);
  return check_launch("gn_finalize");
}

// ------------------------------------------------------------------ layout helpers
// ---- gradient range control for the backward passes.  fp16 gradients underflow below 6e-8 (d(loss)/d(image) of the colour
// losses is loss_scale / (B H W) ~ 1e-6) and overflow above 65504, and every op of the backward chains is linear in the
// incoming gradient, so the entry kernel multiplies by s = 2^e and the exit kernel by 1/s (both exact): e is chosen on the
// device so that max|g| * mult * s lies in [2^T, 2^(T+1)).  gs = {s, 1/s, max slot (float bits; re-armed to 0 here)}.
__global__ void __launch_bounds__(256) absmax_kernel(const float* __restrict__ x, int64_t n, float* __restrict__ gs) {
  pdl_wait();
  float m = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) m = fmaxf(m, fabsf(x[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  // non-negative floats order like their bit patterns (NaN / inf sort above every finite value and end up as s = 1)
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(reinterpret_cast<unsigned*>(gs + 2), __float_as_uint(m));
}
__global__ void grad_scale_finalize_kernel(float* __restrict__ gs, float mult, int target_log2) {
  pdl_wait();
  const float m = gs[2] * mult;
  float sc = 1.f;
  if (m > 0.f && m < INFINITY) {
    int e;
    frexpf(m, &e);                     // m = f * 2^e, f in [0.5, 1)
    int k = target_log2 + 1 - e;       // m * 2^k in [2^T, 2^(T+1))
    k = k > 120 ? 120 : (k < -120 ? -120 : k);
    sc = ldexpf(1.f, k);
  }
  gs[0] = sc; gs[1] = 1.f / sc; gs[2] = 0.f;
}
int grad_scale_launch(const float* x, int64_t n, float* gs, float mult, cudaStream_t st) {
  static const int target = getenv("B2E_GRAD_LOG2") ? atoi(getenv("B2E_GRAD_LOG2")) : 2;
  int grid = (int)((n + 1023) / 1024);
  if (grid > kNumSMs * 8) grid = kNumSMs * 8;
  launch_pdl(absmax_kernel, dim3(grid), dim3(256), 0, st, x, n, gs);
  int rc = check_launch("absmax");
  if (rc) return rc;
  launch_pdl(grad_scale_finalize_kernel, dim3(1), dim3(1), 0, st, gs, mult, target);
  return check_launch("grad_scale_finalize");
}

__global__ void pack_input_kernel(const float* __restrict__ x, f16* __restrict__ out, int B, int C,
                                  int HW, int cpad, const float* __restrict__ gs) {
  pdl_wait();
  const float sc = gs ? gs[0] : 1.f;
  const int64_t total = (int64_t)B * HW;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < total;
       p += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = p / HW, q = p % HW;
    float f[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int c = 0; c < C && c < 8; ++c) f[c] = x[(b * C + c) * HW + q] * sc;
    uint4* o = reinterpret_cast<uint4*>(out + p * cpad);
    o[0] = pack8(f);
    const uint4 z = make_uint4(0, 0, 0, 0);
    for (int i = 1; i < cpad / 8; ++i) o[i] = z;
  }
}

// im2col variant: one thread per pixel gathers its 9 x C neighbourhood (coalesced across the warp, neighbours hit
// L1) and writes the pixel's 64 channels (128 B)
// mask / shift: the optional input transform (1 - mask * x, then (v - shift) / scale) of pack_input_launch; none of it
// is evaluated without them, so the plain packing keeps its arithmetic
template <int C>
__global__ void __launch_bounds__(256) pack_input_im2col_kernel(const float* __restrict__ x, f16* __restrict__ out, int B,
                                                                int H, int W, int planes, const float* __restrict__ shift,
                                                                const float* __restrict__ scale, const float* __restrict__ mask,
                                                                int mask_batched) {
  pdl_wait();
  const int HW = H * W;
  const int64_t total = (int64_t)B * HW;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < total; p += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(p / HW), q = (int)(p % HW), h = q / W, w = q % W;
    float f[64];
#pragma unroll
    for (int k = 0; k < 64; ++k) f[k] = 0.f;
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      const int hh = h + t / 3 - 1, ww = w + t % 3 - 1;
      const bool in = hh >= 0 && hh < H && ww >= 0 && ww < W;
#pragma unroll
      for (int c = 0; c < C; ++c)
        if (in) {
          float v = __ldg(x + ((int64_t)b * C + c) * HW + hh * W + ww);
          if (mask) v = __fsub_rn(1.f, __fmul_rn(__ldg(mask + ((int64_t)(mask_batched ? b : 0) * C + c) * HW + hh * W + ww), v));
          if (shift) v = __fdiv_rn(__fsub_rn(v, __ldg(shift + c)), __ldg(scale + c));
          f[t * C + c] = v;
        }
    }
    uint4* o = reinterpret_cast<uint4*>(out + p * 64 * planes);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint4 hv = pack8(f + 8 * j);
      o[j] = hv;
      if (planes == 3) o[16 + j] = hv;
    }
    if (planes == 3) {   // split-f16 (fp32-accurate mode): [hi | lo | hi]
#pragma unroll
      for (int k = 0; k < 64; ++k) f[k] = __fsub_rn(f[k], f16_to_float(float_to_f16(f[k])));
#pragma unroll
      for (int j = 0; j < 8; ++j) o[8 + j] = pack8(f + 8 * j);
    }
  }
}

int pack_input_launch(const float* x, f16* out, int B, int C, int H, int W, int cpad, bool im2col, cudaStream_t st,
                      int planes, const float* gs, const float* shift, const float* scale, const float* mask, int mask_batched) {
  B2E_REQUIRE(im2col || (!shift && !mask), B2E_UNSUPPORTED_SHAPE, "pack_input: the input transform needs the im2col layout");
  B2E_REQUIRE(!shift == !scale, B2E_INVALID_ARG, "pack_input: shift and scale go together");
  const int HW = H * W;
  int64_t total = (int64_t)B * HW;
  int grid = (int)((total + 255) / 256);
  if (grid > kNumSMs * 16) grid = kNumSMs * 16;
  if (im2col) {
    B2E_REQUIRE(9 * C <= 64 && cpad == 64 && !gs, B2E_UNSUPPORTED_SHAPE, "pack_input: im2col needs 9*C <= 64 (and takes no gradient scale)");
    switch (C) {
      case 1: launch_pdl(pack_input_im2col_kernel<1>, dim3(grid), dim3(256), 0, st, x, out, B, H, W, planes, shift, scale, mask, mask_batched); break;
      case 3: launch_pdl(pack_input_im2col_kernel<3>, dim3(grid), dim3(256), 0, st, x, out, B, H, W, planes, shift, scale, mask, mask_batched); break;
      case 4: launch_pdl(pack_input_im2col_kernel<4>, dim3(grid), dim3(256), 0, st, x, out, B, H, W, planes, shift, scale, mask, mask_batched); break;
      default: B2E_REQUIRE(false, B2E_UNSUPPORTED_SHAPE, "pack_input: im2col supports 1, 3 or 4 input channels (got %d)", C);
    }
    return check_launch("pack_input_im2col");
  }
  B2E_REQUIRE(C <= 8 && cpad % 8 == 0, B2E_UNSUPPORTED_SHAPE, "pack_input: in_channels must be <= 8");
  B2E_REQUIRE(planes == 1, B2E_UNSUPPORTED_SHAPE, "pack_input: split-f16 output needs the im2col layout");
  launch_pdl(pack_input_kernel, dim3(grid), dim3(256), 0, st, x, out, B, C, HW, cpad, gs);
  return check_launch("pack_input");
}

__global__ void upsample2x_kernel(const uint4* __restrict__ in, uint4* __restrict__ out, int N, int H,
                                  int W, int C8) {
  pdl_wait();
  const int64_t total = (int64_t)N * (2 * H) * (2 * W) * C8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C8);
    int64_t r = i / C8;
    const int wo = (int)(r % (2 * W)); r /= (2 * W);
    const int ho = (int)(r % (2 * H));
    const int n = (int)(r / (2 * H));
    out[i] = __ldg(in + (((int64_t)n * H + (ho >> 1)) * W + (wo >> 1)) * C8 + c);
  }
}

int upsample2x_launch(const f16* in, f16* out, int N, int H, int W, int C, cudaStream_t st) {
  B2E_REQUIRE(C % 8 == 0, B2E_UNSUPPORTED_SHAPE, "upsample: C %% 8 != 0");
  int64_t total = (int64_t)N * 4 * H * W * (C / 8);
  int grid = (int)((total + 255) / 256);
  if (grid > kNumSMs * 32) grid = kNumSMs * 32;
  launch_pdl(upsample2x_kernel, dim3(grid), dim3(256), 0, st, (const uint4*)in, (uint4*)out, N, H, W, C / 8);
  return check_launch("upsample2x");
}

// ------------------------------------------------------------------ timestep embedding
// sinusoidal embedding -> linear_1 -> SiLU -> linear_2 -> SiLU (the per-resnet projections all consume
// silu(temb)).  Grid (dim / 32, B): every block recomputes the cheap first layer of its sample and produces 32
// outputs of the second, so the 1 MB of linear_2 weights is spread over ~128 blocks instead of B.
constexpr int kTembSlice = 32;
__global__ void __launch_bounds__(256) temb_mlp_kernel(TembArgs a) {
  pdl_wait();
  pdl_trigger();
  extern __shared__ float sm[];
  float* emb = sm;             // [dim0]
  float* hid = sm + a.dim0;    // [dim]
  const int b = blockIdx.y, tid = threadIdx.x;
  const int half = a.dim0 / 2;
  const float t = (float)a.timesteps[b];
  for (int i = tid; i < half; i += blockDim.x) {
    const float ex = -logf(10000.f) * (float)i / ((float)half - a.freq_shift);
    const float v = t * expf(ex);
    const float sv = sinf(v), cv = cosf(v);
    if (a.flip) { emb[i] = cv; emb[half + i] = sv; } else { emb[i] = sv; emb[half + i] = cv; }
  }
  __syncthreads();
  const int warp = tid >> 5, lane = tid & 31, nw = blockDim.x >> 5;
  // four outputs per warp iteration: their weight loads are independent, so the L2 latency is paid once per
  // four rows instead of once per row (this loop is latency-bound)
  for (int o0 = warp * 4; o0 < a.dim; o0 += nw * 4) {
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int i = lane; i < a.dim0; i += 32) {
      const float e = emb[i];
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (o0 + u < a.dim) acc[u] += __ldg(a.w1 + (int64_t)(o0 + u) * a.dim0 + i) * e;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) acc[u] = warp_sum(acc[u]);
    if (lane < 4 && o0 + lane < a.dim) {
      const float y = (lane == 0 ? acc[0] : lane == 1 ? acc[1] : lane == 2 ? acc[2] : acc[3]) + a.b1[o0 + lane];
      hid[o0 + lane] = y / (1.f + expf(-y));
    }
  }
  __syncthreads();
  const int o_end = min(a.dim, (int)(blockIdx.x + 1) * kTembSlice);
  for (int o0 = blockIdx.x * kTembSlice + warp * 4; o0 < o_end; o0 += nw * 4) {
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int i = lane; i < a.dim; i += 32) {
      const float hv = hid[i];
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (o0 + u < o_end) acc[u] += __ldg(a.w2 + (int64_t)(o0 + u) * a.dim + i) * hv;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) acc[u] = warp_sum(acc[u]);
    if (lane < 4 && o0 + lane < o_end) {
      const float y = (lane == 0 ? acc[0] : lane == 1 ? acc[1] : lane == 2 ? acc[2] : acc[3]) + a.b2[o0 + lane];
      a.act[(int64_t)b * a.dim + o0 + lane] = y / (1.f + expf(-y));
    }
  }
}

// proj[b][o] = wp[o] . act[b] + bp[o]   (warp per output; the weight row is read once and reused for every sample)
// PER = weight elements per lane held in registers: 16 covers dim <= 512 (DDPM / LDM: ~50 registers, five blocks per
// SM; the 64-wide instantiation needs 150 registers = one block per SM, six waves over the ~900 blocks)
constexpr int kTembMaxPerLane = 64;   // dim <= 2048 (SD: 1280)
template <int PER>
__global__ void __launch_bounds__(256) temb_proj_kernel(TembArgs a) {
  pdl_wait();
  pdl_trigger();
  const int o = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (o >= a.sumC) return;
  float w[PER];
  const int per = (a.dim + 31) / 32;
#pragma unroll
  for (int j = 0; j < PER; ++j)
    if (j < per) { const int i = lane + 32 * j; w[j] = i < a.dim ? __ldg(a.wp + (int64_t)o * a.dim + i) : 0.f; }
  const float bias = a.bp[o];
  for (int b0 = 0; b0 < a.B; b0 += 4) {   // four samples per iteration: independent loads / reductions in flight
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (b0 + u < a.B) {
        const float* x = a.act + (int64_t)(b0 + u) * a.dim;
#pragma unroll
        for (int j = 0; j < PER; ++j)
          if (j < per) { const int i = lane + 32 * j; if (i < a.dim) acc[u] += w[j] * x[i]; }
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) acc[u] = warp_sum(acc[u]);
    if (lane < 4 && b0 + lane < a.B)
      a.proj[(int64_t)(b0 + lane) * a.sumC + o] = (lane == 0 ? acc[0] : lane == 1 ? acc[1] : lane == 2 ? acc[2] : acc[3]) + bias;
  }
}

int temb_launch(const TembArgs& a, cudaStream_t st) {
  B2E_REQUIRE(a.dim <= 32 * kTembMaxPerLane, B2E_UNSUPPORTED_SHAPE, "temb: embedding width %d > %d", a.dim,
              32 * kTembMaxPerLane);
  launch_pdl(temb_mlp_kernel, dim3((a.dim + kTembSlice - 1) / kTembSlice, a.B), dim3(256),
             (a.dim0 + a.dim) * sizeof(float), st, a);
  int rc = check_launch("temb_mlp");
  if (rc) return rc;
  if (a.dim <= 32 * 16) launch_pdl(temb_proj_kernel<16>, dim3((a.sumC + 7) / 8), dim3(256), 0, st, a);
  else launch_pdl(temb_proj_kernel<kTembMaxPerLane>, dim3((a.sumC + 7) / 8), dim3(256), 0, st, a);
  return check_launch("temb_proj");
}

// ------------------------------------------------------------------ tensor-core attention helpers
// one warp per row: logits (f16) * scale -> softmax in fp32 -> probabilities (f16), in place.
// 16-byte accesses: lane l owns the 8-value chunks l, l + 32, ... of the row (T % 256 == 0: no tail).
template <int CH>   // chunks per lane = T / 256
__global__ void __launch_bounds__(256) softmax_rows_vec_kernel(f16* __restrict__ s, int64_t rows, float scale) {
  pdl_wait();
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  uint4* r = reinterpret_cast<uint4*>(s + row * (CH * 256));
  float v[CH][8];
  uint4 raw[CH];
#pragma unroll
  for (int i = 0; i < CH; ++i) raw[i] = __ldcs(r + lane + 32 * i);
  float m = -INFINITY;
#pragma unroll
  for (int i = 0; i < CH; ++i) {
    unpack8(raw[i], v[i]);
#pragma unroll
    for (int j = 0; j < 8; ++j) { v[i][j] *= scale; m = fmaxf(m, v[i][j]); }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < CH; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) { v[i][j] = __expf(v[i][j] - m); sum += v[i][j]; }
  sum = warp_sum(sum);
  const float inv = 1.f / sum;
#pragma unroll
  for (int i = 0; i < CH; ++i) {
#pragma unroll
    for (int j = 0; j < 8; ++j) v[i][j] *= inv;
    r[lane + 32 * i] = pack8(v[i]);
  }
}

__global__ void __launch_bounds__(256) softmax_rows_kernel(f16* __restrict__ s, int64_t rows, int T, float scale) {
  pdl_wait();
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  f16* r = s + row * T;
  float v[32];   // T <= 1024 -> at most 32 values per lane
  const int per = T / 32;
  float m = -INFINITY;
  for (int i = 0; i < per; ++i) { v[i] = f16_to_float(r[lane + 32 * i]) * scale; m = fmaxf(m, v[i]); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  float sum = 0.f;
  for (int i = 0; i < per; ++i) { v[i] = __expf(v[i] - m); sum += v[i]; }
  sum = warp_sum(sum);
  const float inv = 1.f / sum;
  for (int i = 0; i < per; ++i) r[lane + 32 * i] = float_to_f16(v[i] * inv);
}

int softmax_rows_launch(f16* s, int64_t rows, int T, float scale, cudaStream_t st) {
  B2E_REQUIRE((T % 32 == 0 && T <= 1024) || T == 2048 || T == 4096, B2E_UNSUPPORTED_SHAPE,
              "softmax: unsupported row length %d", T);
  const dim3 grid((unsigned)((rows + 7) / 8));
  switch (T) {
    case 2048: launch_pdl(softmax_rows_vec_kernel<8>, grid, dim3(256), 0, st, s, rows, scale); break;
    case 4096: launch_pdl(softmax_rows_vec_kernel<16>, grid, dim3(256), 0, st, s, rows, scale); break;
    case 256: launch_pdl(softmax_rows_vec_kernel<1>, grid, dim3(256), 0, st, s, rows, scale); break;
    case 512: launch_pdl(softmax_rows_vec_kernel<2>, grid, dim3(256), 0, st, s, rows, scale); break;
    case 768: launch_pdl(softmax_rows_vec_kernel<3>, grid, dim3(256), 0, st, s, rows, scale); break;
    case 1024: launch_pdl(softmax_rows_vec_kernel<4>, grid, dim3(256), 0, st, s, rows, scale); break;
    default: launch_pdl(softmax_rows_kernel, grid, dim3(256), 0, st, s, rows, T, scale);
  }
  return check_launch("softmax_rows");
}

// 32x32 smem-tiled transpose of the V columns of qkv
__global__ void transpose_v_kernel(const f16* __restrict__ qkv, f16* __restrict__ vt, int T, int C) {
  pdl_wait();
  __shared__ f16 tile[32][33];
  const int n = blockIdx.z, t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const f16* src = qkv + ((int64_t)n * T) * 3 * C + 2 * C;
  for (int i = threadIdx.y; i < 32; i += blockDim.y)
    tile[i][threadIdx.x] = src[(int64_t)(t0 + i) * 3 * C + c0 + threadIdx.x];
  __syncthreads();
  f16* dst = vt + (int64_t)n * C * T;
  for (int i = threadIdx.y; i < 32; i += blockDim.y)
    dst[(int64_t)(c0 + i) * T + t0 + threadIdx.x] = tile[threadIdx.x][i];
}

int transpose_v_launch(const f16* qkv, f16* vt, int N, int T, int C, cudaStream_t st) {
  B2E_REQUIRE(T % 32 == 0 && C % 32 == 0, B2E_UNSUPPORTED_SHAPE, "transpose_v: T and C must be multiples of 32");
  launch_pdl(transpose_v_kernel, dim3(dim3(T / 32, C / 32, N)), dim3(dim3(32, 8)), 0, st, qkv, vt, T, C);
  return check_launch("transpose_v");
}

// ------------------------------------------------------------------ transformer-block kernels (SD UNet2DConditionModel)
// LayerNorm over the channels of every token (f16 NHWC rows of C channels, C % 8 == 0, C <= 2048): one warp per token,
// the row lives in registers between the two passes
// CPL = 16-byte chunks per lane: the register array is sized for the row width (a fixed 8-chunk array costs ~100 registers
// and a third of the occupancy on 320-channel rows; the kernel is latency-bound: one row per warp)
template <int CPL>
__global__ void __launch_bounds__(256) layernorm_rows_kernel(const f16* __restrict__ x, f16* __restrict__ y,
                                                             const float* __restrict__ gamma, const float* __restrict__ beta,
                                                             int64_t rows, int C, float eps) {
  pdl_wait();
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const uint4* xr = reinterpret_cast<const uint4*>(x + row * C);
  uint4* yr = reinterpret_cast<uint4*>(y + row * C);
  const int chunks = C >> 3;
  float v[CPL][8];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < CPL; ++i) {
    const int ch = lane + 32 * i;
    if (ch < chunks) {
      unpack8(__ldg(xr + ch), v[i]);
#pragma unroll
      for (int j = 0; j < 8; ++j) sum += v[i][j];
    }
  }
  sum = warp_sum(sum);
  const float mean = sum / (float)C;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < CPL; ++i) {
    const int ch = lane + 32 * i;
    if (ch < chunks) {
#pragma unroll
      for (int j = 0; j < 8; ++j) { const float d = v[i][j] - mean; sq += d * d; }
    }
  }
  sq = warp_sum(sq);
  const float rstd = rsqrtf(sq / (float)C + eps);
#pragma unroll
  for (int i = 0; i < CPL; ++i) {
    const int ch = lane + 32 * i;
    if (ch < chunks) {
      float o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = (v[i][j] - mean) * rstd * __ldg(gamma + ch * 8 + j) + __ldg(beta + ch * 8 + j);
      yr[ch] = pack8(o);
    }
  }
}

__global__ void layernorm_rows_split_kernel(const f16* __restrict__ x, f16* __restrict__ y, const float* __restrict__ gamma,
                                            const float* __restrict__ beta, int64_t rows, int C, float eps);

int layernorm_rows_launch(const f16* x, f16* y, const float* gamma, const float* beta, int64_t rows, int C, float eps,
                          cudaStream_t st, int planes) {
  if (planes == 3) {
    B2E_REQUIRE(C % 8 == 0 && C <= 2048, B2E_UNSUPPORTED_SHAPE, "layernorm: C = %d (multiple of 8, <= 2048)", C);
    launch_pdl(layernorm_rows_split_kernel, dim3((unsigned)((rows + 7) / 8)), dim3(256), 0, st, x, y, gamma, beta, rows, C, eps);
    return check_launch("layernorm_rows_split");
  }
  B2E_REQUIRE(C % 8 == 0 && C <= 2048, B2E_UNSUPPORTED_SHAPE, "layernorm: unsupported width %d", C);
  const dim3 grid((unsigned)((rows + 7) / 8));
  const int cpl = (C / 8 + 31) / 32;
  switch (cpl) {
    case 1: launch_pdl(layernorm_rows_kernel<1>, grid, dim3(256), 0, st, x, y, gamma, beta, rows, C, eps); break;
    case 2: launch_pdl(layernorm_rows_kernel<2>, grid, dim3(256), 0, st, x, y, gamma, beta, rows, C, eps); break;
    case 3: launch_pdl(layernorm_rows_kernel<3>, grid, dim3(256), 0, st, x, y, gamma, beta, rows, C, eps); break;
    case 4: launch_pdl(layernorm_rows_kernel<4>, grid, dim3(256), 0, st, x, y, gamma, beta, rows, C, eps); break;
    case 5: launch_pdl(layernorm_rows_kernel<5>, grid, dim3(256), 0, st, x, y, gamma, beta, rows, C, eps); break;
    default: launch_pdl(layernorm_rows_kernel<8>, grid, dim3(256), 0, st, x, y, gamma, beta, rows, C, eps); break;
  }
  return check_launch("layernorm_rows");
}

// ---- CLIP text encoder helpers
// (planes = 3: split-f16 rows [hi | lo | hi] of D channels each, value hi + lo, as layernorm_rows_split_kernel)
// token + position embedding: ids int64 [B][L] -> x f16 [B][Lpad][D] (rows >= L zero); the sum is taken in fp32
__global__ void __launch_bounds__(256) clip_embed_kernel(const int64_t* __restrict__ ids, const float* __restrict__ tok,
                                                         const float* __restrict__ pos, f16* __restrict__ out, int B, int L,
                                                         int Lpad, int D8, int vocab, int planes) {
  pdl_wait();
  const int64_t total = (int64_t)B * Lpad * D8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(i % D8);
    const int l = (int)((i / D8) % Lpad);
    const int b = (int)(i / ((int64_t)D8 * Lpad));
    float f[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (l < L) {
      int64_t id = ids[(int64_t)b * L + l];
      id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
      const float4* t = reinterpret_cast<const float4*>(tok + (id * D8 + s) * 8);
      const float4* q = reinterpret_cast<const float4*>(pos + ((int64_t)l * D8 + s) * 8);
      const float4 t0 = __ldg(t), t1 = __ldg(t + 1), q0 = __ldg(q), q1 = __ldg(q + 1);
      f[0] = t0.x + q0.x; f[1] = t0.y + q0.y; f[2] = t0.z + q0.z; f[3] = t0.w + q0.w;
      f[4] = t1.x + q1.x; f[5] = t1.y + q1.y; f[6] = t1.z + q1.z; f[7] = t1.w + q1.w;
    }
    const uint4 hi = pack8(f);
    if (planes == 3) {
      const int64_t r = i / D8;                    // token row
      uint4* o = reinterpret_cast<uint4*>(out) + r * 3 * D8 + s;
      float l[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) l[j] = __fsub_rn(f[j], f16_to_float(float_to_f16(f[j])));
      o[0] = hi; o[D8] = pack8(l); o[2 * D8] = hi;
    } else {
      *reinterpret_cast<uint4*>(out + i * 8) = hi;
    }
  }
}

int clip_embed_launch(const int64_t* ids, const float* tok, const float* pos, f16* out, int B, int L, int Lpad, int D, int vocab,
                      cudaStream_t st, int planes) {
  B2E_REQUIRE(D % 8 == 0 && L <= Lpad && (planes == 1 || planes == 3), B2E_UNSUPPORTED_SHAPE, "clip_embed: bad shape");
  const int64_t total = (int64_t)B * Lpad * (D / 8);
  launch_pdl(clip_embed_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st, ids, tok, pos, out, B, L, Lpad, D / 8, vocab,
             planes);
  return check_launch("clip_embed");
}

// quick_gelu: x * sigmoid(1.702 x), in place capable
__global__ void __launch_bounds__(256) quick_gelu_kernel(const uint4* __restrict__ in, uint4* __restrict__ out, int64_t n8) {
  pdl_wait();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
    float f[8];
    unpack8(in[i], f);
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = f[j] / (1.f + __expf(-1.702f * f[j]));
    out[i] = pack8(f);
  }
}

// fp32-accurate quick_gelu on split rows of C channels per plane: hi + lo -> x * sigmoid(1.702 x) in fp32 (exact expf,
// as the split SiLU) -> hi, lo, hi; in place capable
__global__ void __launch_bounds__(256) quick_gelu_split_kernel(const uint4* __restrict__ in, uint4* __restrict__ out, int64_t rows,
                                                               int C8) {
  pdl_wait();
  const int64_t total = rows * C8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / C8;
    const int c = (int)(i % C8);
    const uint4* row = in + r * 3 * C8;
    float f[8], l[8];
    unpack8(row[c], f);
    unpack8(row[C8 + c], l);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float v = f[j] + l[j];
      f[j] = v / (1.f + expf(-1.702f * v));
      l[j] = __fsub_rn(f[j], f16_to_float(float_to_f16(f[j])));
    }
    uint4* orow = out + r * 3 * C8;
    const uint4 hi = pack8(f);
    orow[c] = hi; orow[C8 + c] = pack8(l); orow[2 * C8 + c] = hi;
  }
}

int quick_gelu_launch(const f16* in, f16* out, int64_t numel, cudaStream_t st, int planes, int C) {
  B2E_REQUIRE(numel % 8 == 0, B2E_UNSUPPORTED_SHAPE, "quick_gelu: numel %% 8 != 0");
  if (planes == 3) {
    B2E_REQUIRE(C > 0 && C % 8 == 0 && numel % (3 * (int64_t)C) == 0, B2E_UNSUPPORTED_SHAPE,
                "quick_gelu: %lld elements are not split rows of 3 x %d channels", (long long)numel, C);
    const int64_t rows = numel / (3 * (int64_t)C);
    int64_t g = (rows * (C / 8) + 255) / 256;
    if (g > kNumSMs * 16) g = kNumSMs * 16;
    launch_pdl(quick_gelu_split_kernel, dim3((unsigned)g), dim3(256), 0, st, (const uint4*)in, (uint4*)out, rows, C / 8);
    return check_launch("quick_gelu_split");
  }
  int64_t g = (numel / 8 + 255) / 256;
  if (g > kNumSMs * 16) g = kNumSMs * 16;
  launch_pdl(quick_gelu_kernel, dim3((unsigned)g), dim3(256), 0, st, (const uint4*)in, (uint4*)out, numel / 8);
  return check_launch("quick_gelu");
}

// final LayerNorm output: rows [0, L) of every sequence, f16 [B][Lpad][D] -> fp32 [B][L][D] (planes = 3: hi + lo)
__global__ void __launch_bounds__(256) unpad_rows_f32_kernel(const f16* __restrict__ x, float* __restrict__ out, int B, int L,
                                                             int Lpad, int D, int planes) {
  pdl_wait();
  const int64_t total = (int64_t)B * L * D;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int d = (int)(i % D);
    const int l = (int)((i / D) % L);
    const int b = (int)(i / ((int64_t)D * L));
    const f16* row = x + ((int64_t)b * Lpad + l) * planes * D;
    out[i] = planes == 3 ? f16_to_float(row[d]) + f16_to_float(row[D + d]) : f16_to_float(row[d]);
  }
}

int unpad_rows_f32_launch(const f16* x, float* out, int B, int L, int Lpad, int D, cudaStream_t st, int planes) {
  B2E_REQUIRE(planes == 1 || planes == 3, B2E_INVALID_ARG, "unpad_rows_f32: planes must be 1 or 3");
  const int64_t total = (int64_t)B * L * D;
  launch_pdl(unpad_rows_f32_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st, x, out, B, L, Lpad, D, planes);
  return check_launch("unpad_rows_f32");
}

// fp32-accurate mode: LayerNorm over split-f16 rows ([hi | lo | hi] planes of C channels, value = hi + lo)
__global__ void __launch_bounds__(256) layernorm_rows_split_kernel(const f16* __restrict__ x, f16* __restrict__ y,
                                                                   const float* __restrict__ gamma, const float* __restrict__ beta,
                                                                   int64_t rows, int C, float eps) {
  pdl_wait();
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const uint4* xr = reinterpret_cast<const uint4*>(x + row * 3 * C);
  uint4* yr = reinterpret_cast<uint4*>(y + row * 3 * C);
  const int chunks = C >> 3;
  float v[8][8];   // up to 8 chunks per lane (C <= 2048)
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int ch = lane + 32 * i;
    if (ch < chunks) {
      float l[8];
      unpack8(__ldg(xr + ch), v[i]);
      unpack8(__ldg(xr + chunks + ch), l);
#pragma unroll
      for (int j = 0; j < 8; ++j) { v[i][j] += l[j]; sum += v[i][j]; }
    }
  }
  sum = warp_sum(sum);
  const float mean = sum / (float)C;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int ch = lane + 32 * i;
    if (ch < chunks) {
#pragma unroll
      for (int j = 0; j < 8; ++j) { const float d = v[i][j] - mean; sq += d * d; }
    }
  }
  sq = warp_sum(sq);
  const float rstd = 1.0f / sqrtf(sq / (float)C + eps);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int ch = lane + 32 * i;
    if (ch < chunks) {
      float o[8], l[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        o[j] = (v[i][j] - mean) * rstd * __ldg(gamma + ch * 8 + j) + __ldg(beta + ch * 8 + j);
        l[j] = __fsub_rn(o[j], f16_to_float(float_to_f16(o[j])));
      }
      const uint4 hi = pack8(o);
      yr[ch] = hi; yr[chunks + ch] = pack8(l); yr[2 * chunks + ch] = hi;
    }
  }
}

// fp32-accurate GEGLU on split rows: in planes of 2*inner channels, out planes of inner channels
__global__ void __launch_bounds__(256) geglu_split_kernel(const uint4* __restrict__ in, uint4* __restrict__ out, int64_t rows,
                                                          int inner8) {
  pdl_wait();
  const int64_t total = rows * inner8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / inner8;
    const int c = (int)(i % inner8);
    const uint4* row = in + r * 6 * inner8;       // [hi (2*inner) | lo (2*inner) | hi]
    float a[8], g[8], al[8], gl[8], l[8];
    unpack8(__ldg(row + c), a);
    unpack8(__ldg(row + inner8 + c), g);
    unpack8(__ldg(row + 2 * inner8 + c), al);
    unpack8(__ldg(row + 3 * inner8 + c), gl);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float av = a[j] + al[j], gv = g[j] + gl[j];
      a[j] = av * (0.5f * gv * (1.f + erff(gv * 0.70710678118654752f)));
      l[j] = __fsub_rn(a[j], f16_to_float(float_to_f16(a[j])));
    }
    uint4* orow = out + r * 3 * inner8;
    const uint4 hi = pack8(a);
    orow[c] = hi; orow[inner8 + c] = pack8(l); orow[2 * inner8 + c] = hi;
  }
}

// GEGLU: in [rows][2*inner] -> out [rows][inner] = in[:, :inner] * gelu(in[:, inner:])   (exact erf GELU)
__global__ void __launch_bounds__(256) geglu_kernel(const uint4* __restrict__ in, uint4* __restrict__ out, int64_t rows,
                                                    int inner8) {
  pdl_wait();
  const int64_t total = rows * inner8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / inner8;
    const int c = (int)(i % inner8);
    float a[8], g[8];
    unpack8(__ldg(in + r * 2 * inner8 + c), a);
    unpack8(__ldg(in + r * 2 * inner8 + inner8 + c), g);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] *= 0.5f * g[j] * (1.f + erff(g[j] * 0.70710678118654752f));
    out[i] = pack8(a);
  }
}

int geglu_launch(const f16* in, f16* out, int64_t rows, int inner, cudaStream_t st, int planes) {
  B2E_REQUIRE(inner % 8 == 0, B2E_UNSUPPORTED_SHAPE, "geglu: inner %% 8");
  const int64_t total = rows * (inner / 8);
  int grid = (int)((total + 255) / 256);
  if (grid > kNumSMs * 32) grid = kNumSMs * 32;
  if (planes == 3) {
    launch_pdl(geglu_split_kernel, dim3(grid), dim3(256), 0, st, (const uint4*)in, (uint4*)out, rows, inner / 8);
    return check_launch("geglu_split");
  }
  launch_pdl(geglu_kernel, dim3(grid), dim3(256), 0, st, (const uint4*)in, (uint4*)out, rows, inner / 8);
  return check_launch("geglu");
}

// text conditioning: fp32 [B][L][D] -> f16 [B][Lpad][D], rows >= L zero
__global__ void __launch_bounds__(256) pack_context_kernel(const float* __restrict__ ctx, f16* __restrict__ out, int B, int L,
                                                           int Lpad, int D, int planes) {
  pdl_wait();
  const int64_t total = (int64_t)B * Lpad * D;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int dcol = (int)(i % D);
    const int l = (int)((i / D) % Lpad);
    const int64_t b = i / ((int64_t)D * Lpad);
    const float v = l < L ? ctx[(b * L + l) * D + dcol] : 0.f;
    const f16 hi = float_to_f16(v);
    if (planes == 3) {   // split-f16 rows [hi | lo | hi]
      f16* o = out + (b * Lpad + l) * 3 * D + dcol;
      o[0] = hi; o[D] = float_to_f16(__fsub_rn(v, f16_to_float(hi))); o[2 * D] = hi;
    } else {
      out[i] = hi;
    }
  }
}

int pack_context_launch(const float* ctx, f16* out, int B, int L, int Lpad, int D, cudaStream_t st, int planes) {
  const int64_t total = (int64_t)B * Lpad * D;
  int grid = (int)((total + 255) / 256);
  if (grid > kNumSMs * 16) grid = kNumSMs * 16;
  launch_pdl(pack_context_kernel, dim3(grid), dim3(256), 0, st, ctx, out, B, L, Lpad, D, planes);
  return check_launch("pack_context");
}

// head-major gather for the batched attention GEMMs.  src rows: token (n, t), channels [col0 + h*d, + d) of a row of
// `pitch` channels, t < Tsrc.  dst [N*heads][Tpad][dpad] with zeros for t >= Tsrc and channels >= d.
__global__ void __launch_bounds__(256) gather_heads_kernel(const f16* __restrict__ src, f16* __restrict__ dst, int N, int Tsrc,
                                                           int Tpad, int pitch, int col0, int heads, int d, int dpad) {
  pdl_wait();
  const int d8 = dpad >> 3;
  const int64_t total = (int64_t)N * heads * Tpad * d8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int j = (int)(i % d8);
    const int t = (int)((i / d8) % Tpad);
    const int64_t v = i / ((int64_t)d8 * Tpad);
    const int64_t n = v / heads;
    const int h = (int)(v % heads);
    uint4 val = make_uint4(0, 0, 0, 0);
    if (t < Tsrc && j * 8 < d) val = __ldg(reinterpret_cast<const uint4*>(src + (n * Tsrc + t) * pitch + col0 + h * d + j * 8));
    reinterpret_cast<uint4*>(dst)[i] = val;
  }
}

// transposed variant: dst [N*heads][dpad][Tpad] (V^T), zeros outside
__global__ void gather_heads_T_kernel(const f16* __restrict__ src, f16* __restrict__ dst, int Tsrc, int Tpad, int pitch,
                                      int col0, int heads, int d, int dpad) {
  pdl_wait();
  __shared__ f16 tile[32][33];
  const int v = blockIdx.z, n = v / heads, h = v % heads, t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const f16* s = src + ((int64_t)n * Tsrc) * pitch + col0 + h * d;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int t = t0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (t < Tsrc && c < d) ? s[(int64_t)t * pitch + c] : float_to_f16(0.f);
  }
  __syncthreads();
  f16* dd = dst + (int64_t)v * dpad * Tpad;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) dd[(int64_t)(c0 + i) * Tpad + t0 + threadIdx.x] = tile[threadIdx.x][i];
}

// inverse of gather_heads for the attention output: out[n][t][h*d + c] = oh[n*heads + h][t][c], t < T, c < d
__global__ void __launch_bounds__(256) scatter_heads_kernel(const f16* __restrict__ oh, f16* __restrict__ out, int N, int T,
                                                            int Tpad, int pitch, int heads, int d, int dpad) {
  pdl_wait();
  const int c8 = pitch >> 3;   // the tail [heads*d, pitch) of every row is zero padding
  const int64_t total = (int64_t)N * T * c8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(i % c8);
    const int64_t nt = i / c8;
    const int64_t n = nt / T;
    const int t = (int)(nt % T);
    const int c0 = s * 8;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (c0 < heads * d) {
      const int h = c0 / d, cc = c0 - h * d;   // d % 8 == 0: an 8-channel slot never straddles two heads
      v = __ldg(reinterpret_cast<const uint4*>(oh + (((n * heads + h) * Tpad + t) * (int64_t)dpad + cc)));
    }
    *reinterpret_cast<uint4*>(out + nt * pitch + c0) = v;
  }
}

int gather_heads_launch(const f16* src, f16* dst, int N, int Tsrc, int Tpad, int pitch, int col0, int heads, int d, int dpad,
                        bool transposed, cudaStream_t st) {
  B2E_REQUIRE(d % 8 == 0 && dpad % 64 == 0 && dpad >= d && Tpad % 32 == 0 && Tpad >= Tsrc, B2E_UNSUPPORTED_SHAPE,
              "gather_heads: head_dim %d -> %d, T %d -> %d", d, dpad, Tsrc, Tpad);
  if (transposed) {
    launch_pdl(gather_heads_T_kernel, dim3(Tpad / 32, dpad / 32, N * heads), dim3(32, 8), 0, st, src, dst, Tsrc, Tpad, pitch, col0,
               heads, d, dpad);
    return check_launch("gather_heads_T");
  }
  const int64_t total = (int64_t)N * heads * Tpad * (dpad / 8);
  int grid = (int)((total + 255) / 256);
  if (grid > kNumSMs * 32) grid = kNumSMs * 32;
  launch_pdl(gather_heads_kernel, dim3(grid), dim3(256), 0, st, src, dst, N, Tsrc, Tpad, pitch, col0, heads, d, dpad);
  return check_launch("gather_heads");
}

int scatter_heads_launch(const f16* oh, f16* out, int N, int T, int Tpad, int pitch, int heads, int d, int dpad, cudaStream_t st) {
  B2E_REQUIRE(d % 8 == 0, B2E_UNSUPPORTED_SHAPE, "scatter_heads: head_dim %d", d);
  const int64_t total = (int64_t)N * T * (pitch / 8);
  int grid = (int)((total + 255) / 256);
  if (grid > kNumSMs * 32) grid = kNumSMs * 32;
  launch_pdl(scatter_heads_kernel, dim3(grid), dim3(256), 0, st, oh, out, N, T, Tpad, pitch, heads, d, dpad);
  return check_launch("scatter_heads");
}

// row softmax with masked tail: row length T (<= 1024, T % 32 == 0), only the first `valid` entries take part, the
// rest become 0 (zero-padded keys of the batched attention GEMMs)
__global__ void __launch_bounds__(256) softmax_rows_masked_kernel(f16* __restrict__ s, int64_t rows, int T, int valid, float scale) {
  pdl_wait();
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  f16* r = s + row * T;
  float v[32];
  const int per = T / 32;
  float m = -INFINITY;
  for (int i = 0; i < per; ++i) {
    const int j = lane + 32 * i;
    v[i] = j < valid ? f16_to_float(r[j]) * scale : -INFINITY;
    m = fmaxf(m, v[i]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  float sum = 0.f;
  for (int i = 0; i < per; ++i) { v[i] = (lane + 32 * i) < valid ? __expf(v[i] - m) : 0.f; sum += v[i]; }
  sum = warp_sum(sum);
  const float inv = 1.f / sum;
  for (int i = 0; i < per; ++i) r[lane + 32 * i] = float_to_f16(v[i] * inv);
}

int softmax_rows_masked_launch(f16* s, int64_t rows, int T, int valid, float scale, cudaStream_t st) {
  if (valid == T) return softmax_rows_launch(s, rows, T, scale, st);
  B2E_REQUIRE(T % 32 == 0 && T <= 1024 && valid >= 1 && valid < T, B2E_UNSUPPORTED_SHAPE,
              "masked softmax: unsupported row length %d (valid %d)", T, valid);
  launch_pdl(softmax_rows_masked_kernel, dim3((unsigned)((rows + 7) / 8)), dim3(256), 0, st, s, rows, T, valid, scale);
  return check_launch("softmax_rows_masked");
}

// ------------------------------------------------------------------ backward helpers of the decoder
// gradient of the nearest x2 upsample: dx[n][h][w][c] = sum of the 2x2 block of dy (f16 NHWC, 8 channels per thread)
__global__ void __launch_bounds__(256) downsum2x_kernel(const uint4* __restrict__ dy, uint4* __restrict__ dx, int N, int H, int W,
                                                        int C8) {
  pdl_wait();
  const int64_t total = (int64_t)N * H * W * C8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C8);
    int64_t p = i / C8;
    const int w = (int)(p % W); p /= W;
    const int h = (int)(p % H);
    const int64_t n = p / H;
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int dh = 0; dh < 2; ++dh)
#pragma unroll
      for (int dw = 0; dw < 2; ++dw) {
        float f[8];
        unpack8(__ldg(dy + ((n * 2 * H + 2 * h + dh) * 2 * W + 2 * w + dw) * C8 + c), f);
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] += f[j];
      }
    dx[i] = pack8(acc);
  }
}

int downsum2x_launch(const f16* dy, f16* dx, int N, int H, int W, int C, cudaStream_t st) {
  B2E_REQUIRE(C % 8 == 0, B2E_UNSUPPORTED_SHAPE, "downsum2x: C %% 8");
  const int64_t total = (int64_t)N * H * W * (C / 8);
  int grid = (int)((total + 255) / 256);
  if (grid > kNumSMs * 32) grid = kNumSMs * 32;
  launch_pdl(downsum2x_kernel, dim3(grid), dim3(256), 0, st, (const uint4*)dy, (uint4*)dx, N, H, W, C / 8);
  return check_launch("downsum2x");
}

// batched 2-D transpose of a column window: dst[n][c][r] = src[n][r][col0 + c], r < R, c < Cc (both multiples of 32)
__global__ void transpose_window_kernel(const f16* __restrict__ src, f16* __restrict__ dst, int R, int Cc, int src_pitch,
                                        int col0) {
  pdl_wait();
  __shared__ f16 tile[32][33];
  const int n = blockIdx.z, r0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const f16* s = src + (int64_t)n * R * src_pitch + col0;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) tile[i][threadIdx.x] = s[(int64_t)(r0 + i) * src_pitch + c0 + threadIdx.x];
  __syncthreads();
  f16* d = dst + (int64_t)n * Cc * R;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) d[(int64_t)(c0 + i) * R + r0 + threadIdx.x] = tile[threadIdx.x][i];
}

// 64 x 64 tiles moved as 32-bit words (two adjacent columns): every warp access is 128 contiguous bytes on both sides
// (the 32 x 32 two-byte version ran at 1.9 TB/s on the 4096 x 4096 attention matrices of the decoder backward pass)
__global__ void __launch_bounds__(256) transpose_window64_kernel(const f16* __restrict__ src, f16* __restrict__ dst, int R,
                                                                 int Cc, int src_pitch, int col0) {
  pdl_wait();
  __shared__ uint32_t tile[64][33];
  const int n = blockIdx.z, r0 = blockIdx.x * 64, c0 = blockIdx.y * 64;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 8 warps
  const f16* s = src + (int64_t)n * R * src_pitch + col0 + c0 + 2 * tx;
#pragma unroll
  for (int i = ty; i < 64; i += 8) tile[i][tx] = __ldg(reinterpret_cast<const uint32_t*>(s + (int64_t)(r0 + i) * src_pitch));
  __syncthreads();
  f16* d = dst + (int64_t)n * Cc * R + r0 + 2 * tx;
#pragma unroll
  for (int c = ty; c < 64; c += 8) {
    const uint32_t w0 = tile[2 * tx][c >> 1], w1 = tile[2 * tx + 1][c >> 1];
    const uint32_t o = (c & 1) ? ((w0 >> 16) | (w1 & 0xffff0000u)) : ((w0 & 0xffffu) | (w1 << 16));
    *reinterpret_cast<uint32_t*>(d + (int64_t)(c0 + c) * R) = o;
  }
}

int transpose_window_launch(const f16* src, f16* dst, int N, int R, int Cc, int src_pitch, int col0, cudaStream_t st) {
  B2E_REQUIRE(R % 32 == 0 && Cc % 32 == 0, B2E_UNSUPPORTED_SHAPE, "transpose: R and C must be multiples of 32");
  if (R % 64 == 0 && Cc % 64 == 0 && src_pitch % 2 == 0 && col0 % 2 == 0) {
    launch_pdl(transpose_window64_kernel, dim3(R / 64, Cc / 64, N), dim3(256), 0, st, src, dst, R, Cc, src_pitch, col0);
    return check_launch("transpose_window64");
  }
  launch_pdl(transpose_window_kernel, dim3(R / 32, Cc / 32, N), dim3(32, 8), 0, st, src, dst, R, Cc, src_pitch, col0);
  return check_launch("transpose_window");
}

// softmax backward, one warp per row, in place on dP:  dS = scale * P o (dP - sum_j dP_j P_j)
__global__ void __launch_bounds__(256) softmax_bwd_rows_kernel(const f16* __restrict__ p, f16* __restrict__ dp, int64_t rows,
                                                               int T, float scale) {
  pdl_wait();
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const uint4* pr = reinterpret_cast<const uint4*>(p + row * T);
  uint4* dr = reinterpret_cast<uint4*>(dp + row * T);
  const int chunks = T >> 3;
  float dot = 0.f;
  for (int i = lane; i < chunks; i += 32) {
    float a[8], b[8];
    unpack8(__ldg(pr + i), a);
    unpack8(dr[i], b);
#pragma unroll
    for (int j = 0; j < 8; ++j) dot += a[j] * b[j];
  }
  dot = warp_sum(dot);
  for (int i = lane; i < chunks; i += 32) {
    float a[8], b[8];
    unpack8(__ldg(pr + i), a);
    unpack8(dr[i], b);
#pragma unroll
    for (int j = 0; j < 8; ++j) b[j] = scale * a[j] * (b[j] - dot);
    dr[i] = pack8(b);
  }
}

int softmax_bwd_rows_launch(const f16* p, f16* dp, int64_t rows, int T, float scale, cudaStream_t st) {
  B2E_REQUIRE(T % 8 == 0, B2E_UNSUPPORTED_SHAPE, "softmax backward: T %% 8");
  launch_pdl(softmax_bwd_rows_kernel, dim3((unsigned)((rows + 7) / 8)), dim3(256), 0, st, p, dp, rows, T, scale);
  return check_launch("softmax_bwd_rows");
}

// backward of (nearest code [straight-through] -> post_quant_conv -> im2col): dcols f16 [B][H][W][64] holds the gradient
// w.r.t. im2col column t*L + c of every pixel; dz[b][k][h][w] = sum_c pq_w[c][k] * sum_t dcols[(h,w) - tap_t][t*L + c]
__global__ void __launch_bounds__(256) vq_col2im_bwd_kernel(const f16* __restrict__ dcols, const float* __restrict__ pq_w,
                                                            float* __restrict__ dz, int B, int L, int H, int W,
                                                            const float* __restrict__ gs, const float* __restrict__ mask,
                                                            int mask_batched) {
  pdl_wait();
  const float unscale = gs ? gs[1] : 1.f;
  const int64_t total = (int64_t)B * H * W;
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= total) return;
  const int HW = H * W;
  const int b = (int)(p / HW), q = (int)(p % HW), h = q / W, w = q % W;
  float g[4] = {0.f, 0.f, 0.f, 0.f};
  for (int t = 0; t < 9; ++t) {
    // forward: cols[(hh, ww)][t*L + c] = x[c][hh + t/3 - 1][ww + t%3 - 1]  ->  (hh, ww) = (h, w) - tap
    const int hh = h - (t / 3 - 1), ww = w - (t % 3 - 1);
    if (hh < 0 || hh >= H || ww < 0 || ww >= W) continue;
    const f16* src = dcols + (((int64_t)b * H + hh) * W + ww) * 64 + t * L;
    for (int c = 0; c < L; ++c) g[c] += f16_to_float(src[c]);
  }
  for (int k = 0; k < L; ++k) {
    float acc = 0.f;
    for (int c = 0; c < L; ++c) acc += pq_w[c * L + k] * g[c];
    float v = acc * unscale;
    if (mask) v = -__ldg(mask + ((int64_t)(mask_batched ? b : 0) * L + k) * HW + q) * v;
    dz[((int64_t)b * L + k) * HW + q] = v;
  }
}

int vq_col2im_bwd_launch(const f16* dcols, const float* pq_w, float* dz, int B, int L, int H, int W, cudaStream_t st,
                         const float* gs, const float* mask, int mask_batched) {
  B2E_REQUIRE(L >= 1 && L <= 4 && 9 * L <= 64, B2E_UNSUPPORTED_SHAPE, "vq_col2im_bwd: latent channels %d", L);
  const int64_t total = (int64_t)B * H * W;
  launch_pdl(vq_col2im_bwd_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st, dcols, pq_w, dz, B, L, H, W, gs, mask, mask_batched);
  return check_launch("vq_col2im_bwd");
}

// ------------------------------------------------------------------ VQ front of the decoder
// VQModel.decode: nearest codebook entry per latent pixel (squared Euclidean distance accumulated channel by
// channel with individually rounded operations, first index on ties - the oracle's order), then the 1x1
// post_quant_conv.  z, out: fp32 NCHW (B, L, HW), L <= 4.  Codes are staged through smem in tiles.
constexpr int kVqTile = 1024;
constexpr int kVqLanes = 8;   // threads per latent pixel: each scans every 8th code (stride-L smem reads are conflict-free)
__global__ void __launch_bounds__(256)
vq_quantize_kernel(const float* __restrict__ z, const float* __restrict__ codebook, int n_codes,
                   const float* __restrict__ pq_w, const float* __restrict__ pq_b, float* __restrict__ out, int B, int L,
                   int HW) {
  pdl_wait();
  __shared__ float s_code[kVqTile * 4];
  const int64_t total = (int64_t)B * HW;
  const int sub = threadIdx.x & (kVqLanes - 1);
  const int64_t p = (int64_t)blockIdx.x * (blockDim.x / kVqLanes) + (threadIdx.x / kVqLanes);
  const bool live = p < total;
  const int64_t b = live ? p / HW : 0, q = live ? p % HW : 0;
  float zv[4] = {0.f, 0.f, 0.f, 0.f};
  if (live)
    for (int c = 0; c < L; ++c) zv[c] = z[(b * L + c) * HW + q];
  float best = INFINITY;
  int best_i = 0x7fffffff;
  for (int k0 = 0; k0 < n_codes; k0 += kVqTile) {
    const int nk = min(kVqTile, n_codes - k0);
    __syncthreads();
    for (int i = threadIdx.x; i < nk * L; i += blockDim.x) s_code[i] = codebook[(int64_t)k0 * L + i];
    __syncthreads();
    if (live) {
      for (int k = sub; k < nk; k += kVqLanes) {
        float d = 0.f;
        for (int c = 0; c < L; ++c) {
          const float t = __fsub_rn(zv[c], s_code[k * L + c]);
          const float t2 = __fmul_rn(t, t);
          d = c == 0 ? t2 : __fadd_rn(d, t2);
        }
        if (d < best) { best = d; best_i = k0 + k; }   // ascending k: the lane keeps its FIRST minimum
      }
    }
  }
  // combine the lanes of a pixel: smaller distance wins, ties go to the smaller index (= first index over all codes)
#pragma unroll
  for (int o = 1; o < kVqLanes; o <<= 1) {
    const float od = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
    if (od < best || (od == best && oi < best_i)) { best = od; best_i = oi; }
  }
  if (!live || sub != 0) return;
  float e[4] = {0.f, 0.f, 0.f, 0.f};
  // n_codes == 0: no quantiser (AutoencoderKL.decode: post_quant_conv only)
  for (int c = 0; c < L; ++c) e[c] = n_codes > 0 ? codebook[(int64_t)best_i * L + c] : zv[c];
  for (int c = 0; c < L; ++c) {
    float acc = 0.f;
    for (int k = 0; k < L; ++k) acc += pq_w[c * L + k] * e[k];
    out[(b * L + c) * HW + q] = acc + pq_b[c];
  }
}

int vq_quantize_launch(const float* z, const float* codebook, int n_codes, const float* pq_w, const float* pq_b, float* out,
                       int B, int L, int HW, cudaStream_t st) {
  B2E_REQUIRE(L >= 1 && L <= 4 && n_codes >= 0, B2E_UNSUPPORTED_SHAPE, "vq_quantize: latent channels %d", L);
  const int64_t total = (int64_t)B * HW;
  const int ppb = 256 / kVqLanes;   // latent pixels per block
  launch_pdl(vq_quantize_kernel, dim3((unsigned)((total + ppb - 1) / ppb)), dim3(256), 0, st, z, codebook, n_codes, pq_w, pq_b,
             out, B, L, HW);
  return check_launch("vq_quantize");
}

// quant_conv of the VQ / KL encoders: 1x1 convolution over fp32 NCHW with few channels (Cin, Cout <= 16)
__global__ void __launch_bounds__(256)
pointwise_conv_f32_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ b,
                          float* __restrict__ out, int B, int Cin, int Cout, int HW) {
  pdl_wait();
  const int64_t total = (int64_t)B * HW;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < total; p += (int64_t)gridDim.x * blockDim.x) {
    const int64_t n = p / HW, q = p % HW;
    float v[16];
    for (int c = 0; c < Cin; ++c) v[c] = x[(n * Cin + c) * HW + q];
    for (int o = 0; o < Cout; ++o) {
      float acc = 0.f;
      for (int c = 0; c < Cin; ++c) acc += __ldg(w + o * Cin + c) * v[c];
      out[(n * Cout + o) * HW + q] = acc + __ldg(b + o);
    }
  }
}

int pointwise_conv_f32_launch(const float* x, const float* w, const float* b, float* out, int B, int Cin, int Cout, int HW,
                              cudaStream_t st) {
  B2E_REQUIRE(Cin >= 1 && Cin <= 16 && Cout >= 1 && Cout <= 16, B2E_UNSUPPORTED_SHAPE, "pointwise_conv: %d -> %d channels", Cin, Cout);
  const int64_t total = (int64_t)B * HW;
  int grid = (int)((total + 255) / 256);
  if (grid > kNumSMs * 16) grid = kNumSMs * 16;
  launch_pdl(pointwise_conv_f32_kernel, dim3(grid), dim3(256), 0, st, x, w, b, out, B, Cin, Cout, HW);
  return check_launch("pointwise_conv_f32");
}

// ------------------------------------------------------------------ multi-head layout helpers
// qkv [N][T][3P] (q | k | v blocks of P channels, head h = channels [h*d, h*d + d) of a block, d <= 64) ->
// head-major operands of the batched tensor-core GEMMs: qh, kh [N*heads][T][64] (channels >= d zero) and
// vht [N*heads][64][T] (V^T, rows >= d zero).  "Virtual image" v = n * heads + h.
__global__ void __launch_bounds__(256) split_heads_qk_kernel(const f16* __restrict__ qkv, f16* __restrict__ qh,
                                                             f16* __restrict__ kh, int64_t NT, int T, int P, int heads, int d) {
  pdl_wait();
  const int64_t total = NT * heads * 8;   // (n*T + t, h, 8-channel slot)
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int j = (int)(i & 7);
    const int h = (int)((i >> 3) % heads);
    const int64_t nt = (i >> 3) / heads;
    const int64_t n = nt / T, t = nt % T;
    uint4 q = make_uint4(0, 0, 0, 0), k = q;
    if (j * 8 < d) {
      const f16* src = qkv + nt * 3 * P + h * d + j * 8;
      q = __ldg(reinterpret_cast<const uint4*>(src));
      k = __ldg(reinterpret_cast<const uint4*>(src + P));
    }
    const int64_t o = (((n * heads + h) * T + t) << 6) + j * 8;
    *reinterpret_cast<uint4*>(qh + o) = q;
    *reinterpret_cast<uint4*>(kh + o) = k;
  }
}

// 32x32 smem-tiled transpose: vht[v][c][t] = V[n][t][h*d + c] (c < d), 0 otherwise
__global__ void split_heads_vt_kernel(const f16* __restrict__ qkv, f16* __restrict__ vht, int T, int P, int heads, int d) {
  pdl_wait();
  __shared__ f16 tile[32][33];
  const int v = blockIdx.z, n = v / heads, h = v % heads, t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const f16* src = qkv + ((int64_t)n * T) * 3 * P + 2 * P + h * d;
  for (int i = threadIdx.y; i < 32; i += blockDim.y)
    tile[i][threadIdx.x] = (c0 + (int)threadIdx.x < d) ? src[(int64_t)(t0 + i) * 3 * P + c0 + threadIdx.x] : float_to_f16(0.f);
  __syncthreads();
  f16* dst = vht + (int64_t)v * 64 * T;
  for (int i = threadIdx.y; i < 32; i += blockDim.y)
    dst[(int64_t)(c0 + i) * T + t0 + threadIdx.x] = tile[threadIdx.x][i];
}

// oh [N*heads][T][64] -> out [N][T][P]: out[n][t][h*d + c] = oh[n*heads + h][t][c]; channels [heads*d, P) zeroed
__global__ void __launch_bounds__(256) merge_heads_kernel(const f16* __restrict__ oh, f16* __restrict__ out, int64_t NT,
                                                          int T, int P, int heads, int d) {
  pdl_wait();
  const int slots = P >> 3;
  const int64_t total = NT * slots;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(i % slots);
    const int64_t nt = i / slots;
    const int c0 = s * 8;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (c0 < heads * d) {
      const int h = c0 / d, cc = c0 - h * d;
      const int64_t n = nt / T, t = nt % T;
      v = __ldg(reinterpret_cast<const uint4*>(oh + ((((n * heads + h) * T + t) << 6) + cc)));
    }
    *reinterpret_cast<uint4*>(out + nt * P + c0) = v;
  }
}

int split_heads_launch(const f16* qkv, f16* qh, f16* kh, f16* vht, int N, int T, int P, int heads, int d, cudaStream_t st) {
  B2E_REQUIRE(d % 8 == 0 && d <= 64 && T % 32 == 0 && heads * d <= P, B2E_UNSUPPORTED_SHAPE, "split_heads: head_dim %d, T %d", d, T);
  const int64_t NT = (int64_t)N * T, total = NT * heads * 8;
  int grid = (int)((total + 255) / 256);
  if (grid > kNumSMs * 32) grid = kNumSMs * 32;
  launch_pdl(split_heads_qk_kernel, dim3(grid), dim3(256), 0, st, qkv, qh, kh, NT, T, P, heads, d);
  int rc = check_launch("split_heads_qk");
  if (rc) return rc;
  launch_pdl(split_heads_vt_kernel, dim3(T / 32, 2, N * heads), dim3(32, 8), 0, st, qkv, vht, T, P, heads, d);
  return check_launch("split_heads_vt");
}

int merge_heads_launch(const f16* oh, f16* out, int N, int T, int P, int heads, int d, cudaStream_t st) {
  const int64_t NT = (int64_t)N * T, total = NT * (P / 8);
  int grid = (int)((total + 255) / 256);
  if (grid > kNumSMs * 32) grid = kNumSMs * 32;
  launch_pdl(merge_heads_kernel, dim3(grid), dim3(256), 0, st, oh, out, NT, T, P, heads, d);
  return check_launch("merge_heads");
}

// ------------------------------------------------------------------ attention core
// Block = (image n, head h, 16 queries).  S = Q K^T * d^-1/2 in smem (fp32), softmax, O = P V.
// qkv rows are [q | k | v] blocks of P channels each (P >= C = heads * d; the tail of a block is zero padding),
// out rows have pitch P (the tail is zero-filled by the h == 0 blocks).
constexpr int kAttThreads = 256;
constexpr int kAttQ = 16;
constexpr int kAttKStride = 72;  // f16 per staged key row (64 + pad): uint4-aligned, conflict-free

// Q = queries per block: 16, or 4 when 16-query blocks would leave most SMs idle (8x8 mid-block attention: T = 64)
template <int Q>
__global__ void __launch_bounds__(kAttThreads)
attention_kernel(const f16* __restrict__ qkv, f16* __restrict__ out, int T, int C, int P, int heads) {
  pdl_wait();
  extern __shared__ __align__(16) uint8_t att_smem[];
  const int d = C / heads;
  float* Qs = reinterpret_cast<float*>(att_smem);            // [16][d]
  float* S = Qs + Q * d;                                  // [16][T]
  f16* Ks = reinterpret_cast<f16*>(S + Q * T);         // [256][72]  (phase 3: fp32 partial sums, 32 KB)
  const int qt = blockIdx.x, h = blockIdx.y, n = blockIdx.z, tid = threadIdx.x;
  const int q0 = qt * Q;
  const int64_t row = 3 * (int64_t)P;
  const f16* base = qkv + (int64_t)n * T * row;
  const float scale = rsqrtf((float)d);
  // load Q tile
  for (int i = tid; i < Q * d; i += kAttThreads) {
    const int q = i / d, c = i % d;
    Qs[i] = (q0 + q < T) ? f16_to_float(base[(int64_t)(q0 + q) * row + h * d + c]) : 0.f;
  }
  if (h == 0 && P > C) {   // zero padding of the output pitch
    for (int i = tid; i < Q * (P - C); i += kAttThreads) {
      const int q = i / (P - C), c = i % (P - C);
      if (q0 + q < T) out[((int64_t)n * T + q0 + q) * P + C + c] = float_to_f16(0.f);
    }
  }
  // phase 1: scores, keys staged in pieces of dc = min(64, d) channels
  const int dc = d < 64 ? d : 64, parts = dc >> 3;
  for (int kt = 0; kt < T; kt += kAttThreads) {
    float acc[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) acc[q] = 0.f;
    const int key = kt + tid;
    for (int c0 = 0; c0 < d; c0 += dc) {
      __syncthreads();
      for (int i = tid; i < kAttThreads * parts; i += kAttThreads) {
        const int kk = i / parts, part = i % parts;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (kt + kk < T)
          v = __ldg(reinterpret_cast<const uint4*>(base + (int64_t)(kt + kk) * row + P + h * d + c0 + part * 8));
        *reinterpret_cast<uint4*>(Ks + kk * kAttKStride + part * 8) = v;
      }
      __syncthreads();
      if (key < T) {
        for (int part = 0; part < parts; ++part) {
          float kf[8];
          unpack8(*reinterpret_cast<const uint4*>(Ks + tid * kAttKStride + part * 8), kf);
#pragma unroll
          for (int q = 0; q < Q; ++q) {
            const float4 a = *reinterpret_cast<const float4*>(Qs + q * d + c0 + part * 8);
            const float4 b = *reinterpret_cast<const float4*>(Qs + q * d + c0 + part * 8 + 4);
            acc[q] += a.x * kf[0] + a.y * kf[1] + a.z * kf[2] + a.w * kf[3] + b.x * kf[4] + b.y * kf[5] +
                      b.z * kf[6] + b.w * kf[7];
          }
        }
      }
    }
    if (key < T) {
#pragma unroll
      for (int q = 0; q < Q; ++q) S[q * T + key] = acc[q] * scale;
    }
  }
  __syncthreads();
  // phase 2: softmax rows (warp per row)
  const int warp = tid >> 5, lane = tid & 31;
  for (int q = warp; q < Q; q += kAttThreads / 32) {
    float m = -INFINITY;
    for (int j = lane; j < T; j += 32) m = fmaxf(m, S[q * T + j]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float sum = 0.f;
    for (int j = lane; j < T; j += 32) { const float e = __expf(S[q * T + j] - m); S[q * T + j] = e; sum += e; }
    sum = warp_sum(sum);
    const float inv = 1.f / sum;
    for (int j = lane; j < T; j += 32) S[q * T + j] *= inv;
  }
  __syncthreads();
  // phase 3: O = P V.  A thread owns a channel pair; with few channels per head (d/2 < 256) the keys are split
  // over `groups` thread groups and the partial sums are combined through smem in a fixed order.
  const int half = d >> 1;
  int groups = half < kAttThreads ? kAttThreads / half : 1;
  while (groups > 1 && T % (4 * groups) != 0) groups >>= 1;   // every group takes a multiple of 4 keys
  if (groups > 1) {
    float* red = reinterpret_cast<float*>(Ks);   // [groups][16][d] fp32, <= 32 KB (groups * d <= 512)
    const int cp = tid % half, ks = tid / half;
    if (ks < groups) {
      float ax[Q], ay[Q];
#pragma unroll
      for (int q = 0; q < Q; ++q) ax[q] = ay[q] = 0.f;
      const int per = T / groups;
      const f16* vp = base + 2 * P + h * d + 2 * cp;
      for (int j = ks * per; j < (ks + 1) * per; j += 4) {
        float2 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u)
          v[u] = f16x2_to_float2(__ldg(reinterpret_cast<const f16x2*>(vp + (int64_t)(j + u) * row)));
#pragma unroll
        for (int q = 0; q < Q; ++q) {
          const float4 p = *reinterpret_cast<const float4*>(S + q * T + j);
          ax[q] += p.x * v[0].x + p.y * v[1].x + p.z * v[2].x + p.w * v[3].x;
          ay[q] += p.x * v[0].y + p.y * v[1].y + p.z * v[2].y + p.w * v[3].y;
        }
      }
#pragma unroll
      for (int q = 0; q < Q; ++q)
        *reinterpret_cast<float2*>(red + ((ks * Q + q) * d + 2 * cp)) = make_float2(ax[q], ay[q]);
    }
    __syncthreads();
    for (int i = tid; i < Q * half; i += kAttThreads) {
      const int q = i / half, c2 = i % half;
      float sx = 0.f, sy = 0.f;
      for (int g = 0; g < groups; ++g) {
        const float2 v = *reinterpret_cast<const float2*>(red + ((g * Q + q) * d + 2 * c2));
        sx += v.x; sy += v.y;
      }
      if (q0 + q < T)
        *reinterpret_cast<f16x2*>(out + ((int64_t)n * T + q0 + q) * P + h * d + 2 * c2) = floats_to_f16x2(sx, sy);
    }
    return;
  }
  for (int c0 = 2 * tid; c0 < d; c0 += 2 * kAttThreads) {
    float ax[Q], ay[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) ax[q] = ay[q] = 0.f;
    const f16* vp = base + 2 * P + h * d + c0;
    for (int j = 0; j < T; j += 4) {  // T % 4 == 0 (checked on the host)
      float2 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u)
        v[u] = f16x2_to_float2(__ldg(reinterpret_cast<const f16x2*>(vp + (int64_t)(j + u) * row)));
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        const float4 p = *reinterpret_cast<const float4*>(S + q * T + j);
        ax[q] += p.x * v[0].x + p.y * v[1].x + p.z * v[2].x + p.w * v[3].x;
        ay[q] += p.x * v[0].y + p.y * v[1].y + p.z * v[2].y + p.w * v[3].y;
      }
    }
#pragma unroll
    for (int q = 0; q < Q; ++q)
      if (q0 + q < T)
        *reinterpret_cast<f16x2*>(out + ((int64_t)n * T + q0 + q) * P + h * d + c0) =
            floats_to_f16x2(ax[q], ay[q]);
  }
}

// fp32-accurate mode: the same attention core on split-f16 tensors, all arithmetic in fp32 on the CUDA cores
// (1.3 % of the UNet's FLOPs).  qkv rows are [hi | lo | hi] planes of 3P channels (q | k | v blocks of P), out rows
// [hi | lo | hi] planes of P channels.  Block = (image, head, 16 queries).
__global__ void __launch_bounds__(kAttThreads)
attention_split_kernel(const f16* __restrict__ qkv, f16* __restrict__ out, int T, int C, int P, int heads) {
  pdl_wait();
  extern __shared__ __align__(16) uint8_t att_smem[];
  const int d = C / heads;
  float* Qs = reinterpret_cast<float*>(att_smem);   // [16][d]
  float* S = Qs + kAttQ * d;                         // [16][T]
  const int qt = blockIdx.x, h = blockIdx.y, n = blockIdx.z, tid = threadIdx.x;
  const int q0 = qt * kAttQ;
  const int64_t plane = 3 * (int64_t)P, row = 3 * plane;
  const f16* base = qkv + (int64_t)n * T * row;
  const float scale = 1.0f / sqrtf((float)d);
  for (int i = tid; i < kAttQ * d; i += kAttThreads) {
    const int q = i / d, c = i % d;
    const f16* qp = base + (int64_t)(q0 + q) * row + h * d + c;
    Qs[i] = (q0 + q < T) ? f16_to_float(qp[0]) + f16_to_float(qp[plane]) : 0.f;
  }
  const int64_t orow = 3 * (int64_t)P;
  if (h == 0 && P > C) {   // zero padding of the output pitch (all planes)
    for (int i = tid; i < kAttQ * (P - C) * 3; i += kAttThreads) {
      const int k = i % 3, r = i / 3, q = r / (P - C), c = r % (P - C);
      if (q0 + q < T) out[((int64_t)n * T + q0 + q) * orow + k * P + C + c] = float_to_f16(0.f);
    }
  }
  __syncthreads();
  // scores: a thread owns a key
  for (int key = tid; key < T; key += kAttThreads) {
    float acc[kAttQ];
#pragma unroll
    for (int q = 0; q < kAttQ; ++q) acc[q] = 0.f;
    const f16* kp = base + (int64_t)key * row + P + h * d;
    for (int c0 = 0; c0 < d; c0 += 8) {
      float kf[8], kl[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(kp + c0)), kf);
      unpack8(__ldg(reinterpret_cast<const uint4*>(kp + plane + c0)), kl);
#pragma unroll
      for (int j = 0; j < 8; ++j) kf[j] += kl[j];
#pragma unroll
      for (int q = 0; q < kAttQ; ++q) {
        const float4 a = *reinterpret_cast<const float4*>(Qs + q * d + c0);
        const float4 b = *reinterpret_cast<const float4*>(Qs + q * d + c0 + 4);
        acc[q] += a.x * kf[0] + a.y * kf[1] + a.z * kf[2] + a.w * kf[3] + b.x * kf[4] + b.y * kf[5] + b.z * kf[6] + b.w * kf[7];
      }
    }
#pragma unroll
    for (int q = 0; q < kAttQ; ++q) S[q * T + key] = acc[q] * scale;
  }
  __syncthreads();
  const int warp = tid >> 5, lane = tid & 31;
  for (int q = warp; q < kAttQ; q += kAttThreads / 32) {
    float m = -INFINITY;
    for (int j = lane; j < T; j += 32) m = fmaxf(m, S[q * T + j]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float sum = 0.f;
    for (int j = lane; j < T; j += 32) { const float e = expf(S[q * T + j] - m); S[q * T + j] = e; sum += e; }
    sum = warp_sum(sum);
    const float inv = 1.f / sum;
    for (int j = lane; j < T; j += 32) S[q * T + j] *= inv;
  }
  __syncthreads();
  // O = P V: a thread owns a channel pair
  for (int c0 = 2 * tid; c0 < d; c0 += 2 * kAttThreads) {
    float ax[kAttQ], ay[kAttQ];
#pragma unroll
    for (int q = 0; q < kAttQ; ++q) ax[q] = ay[q] = 0.f;
    const f16* vp = base + 2 * P + h * d + c0;
    for (int j = 0; j < T; j += 4) {
      float2 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float2 vh = f16x2_to_float2(__ldg(reinterpret_cast<const f16x2*>(vp + (int64_t)(j + u) * row)));
        const float2 vl = f16x2_to_float2(__ldg(reinterpret_cast<const f16x2*>(vp + (int64_t)(j + u) * row + plane)));
        v[u] = make_float2(vh.x + vl.x, vh.y + vl.y);
      }
#pragma unroll
      for (int q = 0; q < kAttQ; ++q) {
        const float4 p = *reinterpret_cast<const float4*>(S + q * T + j);
        ax[q] += p.x * v[0].x + p.y * v[1].x + p.z * v[2].x + p.w * v[3].x;
        ay[q] += p.x * v[0].y + p.y * v[1].y + p.z * v[2].y + p.w * v[3].y;
      }
    }
#pragma unroll
    for (int q = 0; q < kAttQ; ++q)
      if (q0 + q < T) {
        f16* o = out + ((int64_t)n * T + q0 + q) * orow + h * d + c0;
        const f16x2 hi = floats_to_f16x2(ax[q], ay[q]);
        const float2 hf = f16x2_to_float2(hi);
        *reinterpret_cast<f16x2*>(o) = hi;
        *reinterpret_cast<f16x2*>(o + P) = floats_to_f16x2(__fsub_rn(ax[q], hf.x), __fsub_rn(ay[q], hf.y));
        *reinterpret_cast<f16x2*>(o + 2 * P) = hi;
      }
  }
}

int attention_split_launch(const f16* qkv, f16* out, int N, int T, int C, int P, int heads, cudaStream_t st) {
  B2E_REQUIRE(heads >= 1 && C % heads == 0 && P >= C && P % 8 == 0, B2E_UNSUPPORTED_SHAPE, "attention: bad head count / pitch");
  const int d = C / heads;
  B2E_REQUIRE(d % 8 == 0 && T % 4 == 0, B2E_UNSUPPORTED_SHAPE, "attention (fp32-accurate): unsupported T=%d head_dim=%d", T, d);
  const size_t smem = sizeof(float) * kAttQ * (d + T);
  B2E_REQUIRE(smem <= 200 * 1024, B2E_UNSUPPORTED_SHAPE, "attention (fp32-accurate): tile does not fit in shared memory");
  static size_t attr = 0;
  if (smem > attr) {
    B2E_CUDA(cudaFuncSetAttribute(attention_split_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr = smem;
  }
  launch_pdl(attention_split_kernel, dim3((T + kAttQ - 1) / kAttQ, heads, N), dim3(kAttThreads), smem, st, qkv, out, T, C, P, heads);
  return check_launch("attention_split");
}

// fp32-accurate mode, any sequence length: flash-style fp32 attention on the CUDA cores (online softmax over 32-key
// tiles, O accumulated in registers).  q / k / v are channel windows of split-f16 tensors ([hi | lo | hi] planes):
// q rows [n][tq] of a tensor with `q_plane` channels per plane at column q_col + h*d, k / v rows [n][tk] of a tensor with
// `k_plane` channels per plane at columns k_col + h*d / v_col + h*d; out rows [n][tq] with o_plane channels per plane.
// Block = (32 queries, head, image).  Causal (CLIP text encoder): query row r sees keys <= min(r, valid_k - 1), and the
// key tiles wholly above the block's diagonal are skipped.
constexpr int kTaQ = 32, kTaK = 32, kTaThreads = 256;
struct TiledAttnArgs {
  const f16* q; const f16* kv; f16* out;
  int Tq, Tk, valid_k, heads, d;
  int q_plane, q_col, k_plane, k_col, v_col, o_plane, o_real;
  int64_t q_img, kv_img, o_img;   // elements between consecutive images
  float scale;
};

template <bool Causal>
__global__ void __launch_bounds__(kTaThreads) attention_split_tiled_kernel(TiledAttnArgs a) {
  pdl_wait();
  extern __shared__ __align__(16) uint8_t ta_smem[];
  const int d = a.d, ds = d + 1;                                  // padded row stride: conflict-free column walks
  float* Qs = reinterpret_cast<float*>(ta_smem);                  // [32][ds]
  float* KV = Qs + kTaQ * ds;                                     // [32][ds]  (K tile, then V tile)
  float* S = KV + kTaK * ds;                                      // [32][33]
  float* rowm = S + kTaQ * (kTaK + 1);                            // [32] running maximum
  float* rowl = rowm + kTaQ;                                      // [32] running sum
  float* rowc = rowl + kTaQ;                                      // [32] rescale factor of the current tile
  const int tid = threadIdx.x, h = blockIdx.y, n = blockIdx.z, q0 = blockIdx.x * kTaQ;
  const f16* qb = a.q + (int64_t)n * a.q_img + a.q_col + h * d;
  const f16* kb = a.kv + (int64_t)n * a.kv_img + a.k_col + h * d;
  const f16* vb = a.kv + (int64_t)n * a.kv_img + a.v_col + h * d;
  const int64_t qrow = 3 * (int64_t)a.q_plane, krow = 3 * (int64_t)a.k_plane;
  for (int i = tid; i < kTaQ * d; i += kTaThreads) {
    const int q = i / d, c = i - q * d;
    float v = 0.f;
    if (q0 + q < a.Tq) { const f16* p = qb + (int64_t)(q0 + q) * qrow + c; v = f16_to_float(p[0]) + f16_to_float(p[a.q_plane]); }
    Qs[q * ds + c] = v * a.scale;
  }
  if (tid < kTaQ) { rowm[tid] = -INFINITY; rowl[tid] = 0.f; }
  // output ownership: column pair cp of query group qg
  const int half = d >> 1;
  const int ngroups = half >= kTaThreads ? 1 : kTaThreads / half;
  const int cp = tid % half, qg = tid / half;
  const int qper = (kTaQ + ngroups - 1) / ngroups;                // queries per group (<= 32)
  const bool owner = qg < ngroups;
  float ox[kTaQ], oy[kTaQ];
#pragma unroll
  for (int i = 0; i < kTaQ; ++i) ox[i] = oy[i] = 0.f;
  __syncthreads();
  // causal: the block's last query row q0 + kTaQ - 1 sees no key past itself (kTaQ == kTaK: tiles align with the diagonal)
  const int k_end = Causal ? min(a.valid_k, q0 + kTaQ) : a.valid_k;
  for (int k0 = 0; k0 < k_end; k0 += kTaK) {
    // ---- K tile -> smem (fp32 = hi + lo)
    for (int i = tid; i < kTaK * d; i += kTaThreads) {
      const int k = i / d, c = i - k * d;
      float v = 0.f;
      if (k0 + k < a.valid_k) { const f16* p = kb + (int64_t)(k0 + k) * krow + c; v = f16_to_float(p[0]) + f16_to_float(p[a.k_plane]); }
      KV[k * ds + c] = v;
    }
    __syncthreads();
    // ---- scores: thread = (query tid / 8, keys (tid % 8) * 4 .. + 3)
    {
      const int q = tid >> 3, kk = (tid & 7) * 4;
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
      const float* qr = Qs + q * ds;
      const float* k0r = KV + kk * ds;
      for (int c = 0; c < d; ++c) {
        const float qv = qr[c];
        s0 += qv * k0r[c]; s1 += qv * k0r[ds + c]; s2 += qv * k0r[2 * ds + c]; s3 += qv * k0r[3 * ds + c];
      }
      // keys this query row may see: the valid prefix, cut at the diagonal for causal attention (every row sees key 0,
      // so the first tile gives each row a finite running maximum)
      const int lim = Causal ? min(a.valid_k, q0 + q + 1) : a.valid_k;
      float* sr = S + q * (kTaK + 1) + kk;
      sr[0] = k0 + kk < lim ? s0 : -INFINITY;
      sr[1] = k0 + kk + 1 < lim ? s1 : -INFINITY;
      sr[2] = k0 + kk + 2 < lim ? s2 : -INFINITY;
      sr[3] = k0 + kk + 3 < lim ? s3 : -INFINITY;
    }
    __syncthreads();
    // ---- online softmax per query row (one warp handles 4 rows; lane = key)
    {
      const int warp = tid >> 5, lane = tid & 31;
      for (int q = warp; q < kTaQ; q += kTaThreads / 32) {
        const float sv = S[q * (kTaK + 1) + lane];
        float mx = sv;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        const float mold = rowm[q], mnew = fmaxf(mold, mx);
        const float pv = sv == -INFINITY ? 0.f : expf(sv - mnew);
        const float ps = warp_sum(pv);
        S[q * (kTaK + 1) + lane] = pv;
        if (lane == 0) {
          const float corr = mold == -INFINITY ? 0.f : expf(mold - mnew);
          rowc[q] = corr; rowm[q] = mnew; rowl[q] = rowl[q] * corr + ps;
        }
      }
    }
    __syncthreads();
    // ---- V tile -> smem (reuses the K buffer)
    for (int i = tid; i < kTaK * d; i += kTaThreads) {
      const int k = i / d, c = i - k * d;
      float v = 0.f;
      if (k0 + k < a.valid_k) { const f16* p = vb + (int64_t)(k0 + k) * krow + c; v = f16_to_float(p[0]) + f16_to_float(p[a.k_plane]); }
      KV[k * ds + c] = v;
    }
    __syncthreads();
    // ---- O = O * corr + P V
    if (owner) {
      for (int c0 = 2 * cp; c0 < d; c0 += 2 * kTaThreads) {   // d <= 512: one pass
#pragma unroll
        for (int i = 0; i < kTaQ; ++i) {
          const int q = qg * qper + i;
          if (i < qper && q < kTaQ) {
            const float corr = rowc[q];
            float ax = ox[i] * corr, ay = oy[i] * corr;
            const float* pr = S + q * (kTaK + 1);
#pragma unroll 8
            for (int k = 0; k < kTaK; ++k) {
              const float pv = pr[k];
              ax += pv * KV[k * ds + c0]; ay += pv * KV[k * ds + c0 + 1];
            }
            ox[i] = ax; oy[i] = ay;
          }
        }
      }
    }
    __syncthreads();
  }
  // ---- normalise and write the split output
  const int64_t orow = 3 * (int64_t)a.o_plane;
  f16* ob = a.out + (int64_t)n * a.o_img + h * d;
  if (owner && 2 * cp < d) {
#pragma unroll
    for (int i = 0; i < kTaQ; ++i) {
      const int q = qg * qper + i;
      if (i < qper && q < kTaQ && q0 + q < a.Tq) {
        const float inv = 1.f / rowl[q];
        const float vx = ox[i] * inv, vy = oy[i] * inv;
        f16* o = ob + (int64_t)(q0 + q) * orow + 2 * cp;
        const f16x2 hi = floats_to_f16x2(vx, vy);
        const float2 hf = f16x2_to_float2(hi);
        *reinterpret_cast<f16x2*>(o) = hi;
        *reinterpret_cast<f16x2*>(o + a.o_plane) = floats_to_f16x2(__fsub_rn(vx, hf.x), __fsub_rn(vy, hf.y));
        *reinterpret_cast<f16x2*>(o + 2 * a.o_plane) = hi;
      }
    }
  }
  if (h == 0 && a.o_plane > a.o_real) {   // zero padding of the output pitch (all planes)
    const int pad = a.o_plane - a.o_real;
    for (int i = tid; i < kTaQ * pad * 3; i += kTaThreads) {
      const int k = i % 3, r = i / 3, q = r / pad, c = r % pad;
      if (q0 + q < a.Tq) a.out[(int64_t)n * a.o_img + (int64_t)(q0 + q) * orow + k * a.o_plane + a.o_real + c] = float_to_f16(0.f);
    }
  }
}

int attention_split_tiled_launch(const f16* q, int q_plane, int q_col, const f16* kv, int k_plane, int k_col, int v_col, f16* out,
                                 int o_plane, int o_real, int N, int Tq, int Tk_rows, int valid_k, int heads, int d, cudaStream_t st,
                                 int causal) {
  B2E_REQUIRE(d % 2 == 0 && d >= 8 && d <= 512 && heads >= 1 && valid_k >= 1 && valid_k <= Tk_rows, B2E_UNSUPPORTED_SHAPE,
              "attention (fp32-accurate, tiled): unsupported head_dim %d / keys %d of %d", d, valid_k, Tk_rows);
  TiledAttnArgs a;
  a.q = q; a.kv = kv; a.out = out; a.Tq = Tq; a.Tk = Tk_rows; a.valid_k = valid_k; a.heads = heads; a.d = d;
  a.q_plane = q_plane; a.q_col = q_col; a.k_plane = k_plane; a.k_col = k_col; a.v_col = v_col; a.o_plane = o_plane; a.o_real = o_real;
  a.q_img = (int64_t)Tq * 3 * q_plane; a.kv_img = (int64_t)Tk_rows * 3 * k_plane; a.o_img = (int64_t)Tq * 3 * o_plane;
  a.scale = 1.0f / sqrtf((float)d);
  const size_t smem = sizeof(float) * ((size_t)(kTaQ + kTaK) * (d + 1) + kTaQ * (kTaK + 1) + 3 * kTaQ);
  static size_t attr[2] = {0, 0};
  const dim3 grid((Tq + kTaQ - 1) / kTaQ, heads, N);
  if (causal) {
    if (smem > attr[1]) {
      B2E_CUDA(cudaFuncSetAttribute(attention_split_tiled_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      attr[1] = smem;
    }
    launch_pdl(attention_split_tiled_kernel<true>, grid, dim3(kTaThreads), smem, st, a);
    return check_launch("attention_split_tiled_causal");
  }
  if (smem > attr[0]) {
    B2E_CUDA(cudaFuncSetAttribute(attention_split_tiled_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr[0] = smem;
  }
  launch_pdl(attention_split_tiled_kernel<false>, grid, dim3(kTaThreads), smem, st, a);
  return check_launch("attention_split_tiled");
}

int attention_launch(const f16* qkv, f16* out, int N, int T, int C, int P, int heads, cudaStream_t st) {
  B2E_REQUIRE(heads >= 1 && C % heads == 0 && P >= C && P % 8 == 0, B2E_UNSUPPORTED_SHAPE, "attention: bad head count / pitch");
  const int d = C / heads;
  B2E_REQUIRE(d % 8 == 0 && (d <= 64 || d % 64 == 0) && d <= 1024 && T % 4 == 0 && T <= 4096, B2E_UNSUPPORTED_SHAPE,
              "attention: unsupported T=%d head_dim=%d", T, d);
  // 4-query blocks when 16-query blocks cannot fill the chip (each block re-stages the keys, so only then)
  const bool small = (int64_t)((T + kAttQ - 1) / kAttQ) * heads * N < kNumSMs;
  const int Q = small ? 4 : kAttQ;
  const size_t smem = sizeof(float) * Q * (d + T) + sizeof(f16) * kAttThreads * kAttKStride;
  B2E_REQUIRE(smem <= 200 * 1024, B2E_UNSUPPORTED_SHAPE, "attention: tile does not fit in shared memory");
  static size_t attr[2] = {0, 0};
  if (smem > attr[small]) {
    if (small) B2E_CUDA(cudaFuncSetAttribute(attention_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    else B2E_CUDA(cudaFuncSetAttribute(attention_kernel<kAttQ>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr[small] = smem;
  }
  if (small) launch_pdl(attention_kernel<4>, dim3((T + 3) / 4, heads, N), dim3(kAttThreads), smem, st, qkv, out, T, C, P, heads);
  else launch_pdl(attention_kernel<kAttQ>, dim3((T + kAttQ - 1) / kAttQ, heads, N), dim3(kAttThreads), smem, st, qkv, out, T, C, P, heads);
  return check_launch("attention");
}

}  // namespace b2e
