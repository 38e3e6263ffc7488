// HBM-bound companions of the GEMM kernels: layout conversion, first/last-layer im2col / col2im,
// BatchNorm (finalize, apply + activation, backward reduce / apply), losses, Adam, weight packing.
// All are plain coalesced / vectorised SIMT kernels with warp-shuffle reductions; none stages a
// tensor through an extra HBM round trip beyond the one pass its definition needs.
#include "common.h"
#include "ptx.cuh"

namespace gap {

__device__ __forceinline__ float act_fwd(float v, int act) {
  switch (act) {
    case GAP_ACT_LRELU:
      return v > 0.f ? v : 0.2f * v;
    case GAP_ACT_RELU:
      return fmaxf(v, 0.f);
    case GAP_ACT_TANH:
      return tanhf(v);
    case GAP_ACT_SIGMOID:
      return 1.f / (1.f + __expf(-v));
    default:
      return v;
  }
}

// Grid for a grid-stride kernel whose blocks take `per_block` work items per sweep: at most max_blocks blocks, sized so
// that every sweep is full (a 1.7-sweep launch costs two sweeps; 2048 blocks x 2 full sweeps beat 2368 x 1.73).
static inline int grid_even(long long work, long long per_block, int max_blocks) {
  long long b = (work + per_block - 1) / per_block;
  if (b < 1) b = 1;
  const long long sweeps = (b + max_blocks - 1) / max_blocks;
  return static_cast<int>((b + sweeps - 1) / sweeps);
}

static inline int grid_for(long long work, int block, int max_blocks = 148 * 16) {
  long long g = (work + block - 1) / block;
  if (g < 1) g = 1;
  if (g > max_blocks) g = max_blocks;
  return static_cast<int>(g);
}

// ------------------------------------------------------------------------------------------------
// layout conversion (model boundary only: 1..8 channels)
// ------------------------------------------------------------------------------------------------
__global__ void nchw_f32_to_nhwc_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ out,
                                             int n, int c, long long hw, long long ld) {
  const long long total = static_cast<long long>(n) * hw;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long img = i / hw, pix = i - img * hw;
    for (int ch = 0; ch < c; ++ch)
      out[i * ld + ch] = __float2bfloat16(x[(img * c + ch) * hw + pix]);
  }
}

// 1..4 channels into 4-slot pixels (the image inputs of both networks), 4 pixels per thread: C 16-byte plane loads and
// one 32-byte store instead of 4C scalar loads and 4C two-byte stores (the scalar version ran at 2 TB/s).  Slots >= C are
// written as zero.
template <int C>
__global__ void nchw_f32_to_nhwc4_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ out, long long hw4,
                                              long long total4) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total4;
       i += (long long)gridDim.x * blockDim.x) {
    const long long img = i / hw4, q = i - img * hw4;
    const float4* base = reinterpret_cast<const float4*>(x) + img * C * hw4 + q;
    float4 v[4];
#pragma unroll
    for (int ch = 0; ch < 4; ++ch) v[ch] = ch < C ? __ldg(base + ch * hw4) : make_float4(0.f, 0.f, 0.f, 0.f);
    uint4 lo, hi;
    lo.x = pack_bf16x2(v[0].x, v[1].x);
    lo.y = pack_bf16x2(v[2].x, v[3].x);
    lo.z = pack_bf16x2(v[0].y, v[1].y);
    lo.w = pack_bf16x2(v[2].y, v[3].y);
    hi.x = pack_bf16x2(v[0].z, v[1].z);
    hi.y = pack_bf16x2(v[2].z, v[3].z);
    hi.z = pack_bf16x2(v[0].w, v[1].w);
    hi.w = pack_bf16x2(v[2].w, v[3].w);
    uint4* o = reinterpret_cast<uint4*>(out + i * 16);
    o[0] = lo;
    o[1] = hi;
  }
}

template <typename T>
__global__ void nhwc_to_nchw_f32_kernel(const T* __restrict__ x, float* __restrict__ out, int n, int c,
                                        long long hw, long long ld, int c_total, int c_off) {
  const long long total = static_cast<long long>(n) * hw;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long img = i / hw, pix = i - img * hw;
    for (int ch = 0; ch < c; ++ch)
      out[(img * c_total + c_off + ch) * hw + pix] = static_cast<float>(x[i * ld + ch]);
  }
}

// Tanh backward at the model boundary: dpre[nhwc bf16] = gout[nchw f32] * (1 - y[nhwc f32]^2)
__global__ void tanh_bwd_kernel(const float* __restrict__ gout, const float* __restrict__ y, long long ld_y,
                                __nv_bfloat16* __restrict__ dpre, long long ld_p, int n, int c, long long hw) {
  const long long total = static_cast<long long>(n) * hw;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long img = i / hw, pix = i - img * hw;
    for (int ch = 0; ch < c; ++ch) {
      const float v = y[i * ld_y + ch];
      dpre[i * ld_p + ch] = __float2bfloat16(gout[(img * c + ch) * hw + pix] * (1.f - v * v));
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Generator output backward + L1 loss (train_gan.py:68-70 through Tanh, models.py:186):
//   l1 += sum |fake - real|;  g = dfake_d + l1_scale * sign(fake - real);  dpre = g * (1 - fake^2)
// fake: fp32 NHWC (ld_f), real: fp32 NCHW (the caller's tensor), dfake_d: fp32 NHWC (ld_d, may be
// NULL), dpre: bf16 NHWC (ld_p).  loss_acc[0] accumulates the raw L1 sum in fp64.
// ------------------------------------------------------------------------------------------------
// REAL_U8: `real` is the raw uint8 HWC image [pixel][c]; it is normalised like the dataset does in fp32
// ((x / 255) * 2 - 1, dataset.py:28-29,155-159), so the loss sees exactly the reference's real_B without an fp32 copy.
template <bool REAL_U8>
__global__ void gen_out_bwd_kernel(const float* __restrict__ fake, long long ld_f,
                                   const void* __restrict__ real_v, long long hw,
                                   const float* __restrict__ dfake_d, long long ld_d, float l1_scale,
                                   __nv_bfloat16* __restrict__ dpre, long long ld_p, long long pixels, int c,
                                   double* __restrict__ loss_acc) {
  const float* real = static_cast<const float*>(real_v);
  const unsigned char* real_u8 = static_cast<const unsigned char*>(real_v);
  float part = 0.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < pixels;
       i += (long long)gridDim.x * blockDim.x) {
    const long long img = i / hw, pix = i - img * hw;
    for (int ch = 0; ch < c; ++ch) {
      const float f = fake[i * ld_f + ch];
      const float r = REAL_U8 ? (static_cast<float>(real_u8[i * c + ch]) / 255.f) * 2.f - 1.f
                              : real[(img * c + ch) * hw + pix];
      const float d = f - r;
      part += fabsf(d);
      float g = l1_scale * (d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f));
      if (dfake_d) g += dfake_d[i * ld_d + ch];
      dpre[i * ld_p + ch] = __float2bfloat16(g * (1.f - f * f));
    }
  }
  part = warp_sum(part);
  __shared__ float red[32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) red[wid] = part;
  __syncthreads();
  if (wid == 0) {
    float v = lane < (blockDim.x >> 5) ? red[lane] : 0.f;
    v = warp_sum(v);
    if (lane == 0) atomicAdd(loss_acc, static_cast<double>(v));
  }
}

// The same for the layout the trainer uses (C = 1..4 channels in 4-slot NHWC tensors, hw % 4 == 0): four pixels per
// thread, 128-bit loads of fake / dfake_d, the real image as C 32-bit words (uint8) or C float4 (fp32 planes), two
// 128-bit stores (slots >= C are written as zero, which is what they hold), no per-pixel 64-bit division.  The
// per-pixel scalar kernel above ran at 3.1 TB/s.
template <bool REAL_U8, int C>
__global__ void __launch_bounds__(256) gen_out_bwd_vec_kernel(const float* __restrict__ fake, const void* __restrict__ real_v,
                                                              long long hw, const float* __restrict__ dfake_d, float l1_scale,
                                                              __nv_bfloat16* __restrict__ dpre, long long pixels,
                                                              double* __restrict__ loss_acc) {
  float part = 0.f;
  const long long quads = pixels >> 2;
  for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < quads; q += (long long)gridDim.x * blockDim.x) {
    const long long i = q << 2;
    float4 f[4], dd[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) f[k] = __ldg(reinterpret_cast<const float4*>(fake + (i + k) * 4));
    if (dfake_d) {
#pragma unroll
      for (int k = 0; k < 4; ++k) dd[k] = __ldg(reinterpret_cast<const float4*>(dfake_d + (i + k) * 4));
    }
    float r[4][C];
    if (REAL_U8) {
      const uint32_t* rp = reinterpret_cast<const uint32_t*>(static_cast<const unsigned char*>(real_v) + i * C);
      uint32_t w[C];
#pragma unroll
      for (int k = 0; k < C; ++k) w[k] = __ldg(rp + k);
#pragma unroll
      for (int b = 0; b < 4 * C; ++b)
        r[b / C][b % C] = (static_cast<float>((w[b >> 2] >> (8 * (b & 3))) & 0xffu) / 255.f) * 2.f - 1.f;
    } else {
      const long long img = i / hw, pix = i - img * hw;
      const float* rp = static_cast<const float*>(real_v) + img * C * hw + pix;
#pragma unroll
      for (int ch = 0; ch < C; ++ch) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(rp + ch * hw));
        r[0][ch] = v.x; r[1][ch] = v.y; r[2][ch] = v.z; r[3][ch] = v.w;
      }
    }
    uint32_t pk[8];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float fv[4] = {f[k].x, f[k].y, f[k].z, f[k].w};
      const float dv[4] = {dd[k].x, dd[k].y, dd[k].z, dd[k].w};
      float o[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int ch = 0; ch < C; ++ch) {
        const float d = fv[ch] - r[k][ch];
        part += fabsf(d);
        float g = l1_scale * (d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f));
        if (dfake_d) g += dv[ch];
        o[ch] = g * (1.f - fv[ch] * fv[ch]);
      }
      pk[2 * k] = pack_bf16x2(o[0], o[1]);
      pk[2 * k + 1] = pack_bf16x2(o[2], o[3]);
    }
    uint4* dst = reinterpret_cast<uint4*>(dpre + i * 4);
    dst[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    dst[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
  }
  part = warp_sum(part);
  __shared__ float red[32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) red[wid] = part;
  __syncthreads();
  if (wid == 0) {
    float v = lane < (blockDim.x >> 5) ? red[lane] : 0.f;
    v = warp_sum(v);
    if (lane == 0) atomicAdd(loss_acc, static_cast<double>(v));
  }
}

template <bool REAL_U8>
static void gen_out_bwd_vec_launch(const float* fake, const void* real, int64_t hw, const float* dfake_d, float l1_scale,
                                   void* dpre, int64_t pixels, int c, double* loss_acc, cudaStream_t st) {
  const int grid = grid_for(pixels / 4, 256, 148 * 8);
  __nv_bfloat16* d = static_cast<__nv_bfloat16*>(dpre);
  switch (c) {
    case 1: gen_out_bwd_vec_kernel<REAL_U8, 1><<<grid, 256, 0, st>>>(fake, real, hw, dfake_d, l1_scale, d, pixels, loss_acc); break;
    case 2: gen_out_bwd_vec_kernel<REAL_U8, 2><<<grid, 256, 0, st>>>(fake, real, hw, dfake_d, l1_scale, d, pixels, loss_acc); break;
    case 3: gen_out_bwd_vec_kernel<REAL_U8, 3><<<grid, 256, 0, st>>>(fake, real, hw, dfake_d, l1_scale, d, pixels, loss_acc); break;
    default: gen_out_bwd_vec_kernel<REAL_U8, 4><<<grid, 256, 0, st>>>(fake, real, hw, dfake_d, l1_scale, d, pixels, loss_acc); break;
  }
}

// ------------------------------------------------------------------------------------------------
// BCE-with-logits against a constant target (train_gan.py:42,58,60,67):
//   loss_acc += sum max(x,0) - x*t + log1p(exp(-|x|));  dlogit = grad_scale * (sigmoid(x) - t)
// ------------------------------------------------------------------------------------------------
__global__ void bce_logits_const_kernel(const float* __restrict__ x, long long count, float t,
                                        float grad_scale, __nv_bfloat16* __restrict__ dx, long long ld_dx,
                                        double* __restrict__ loss_acc) {
  float part = 0.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < count;
       i += (long long)gridDim.x * blockDim.x) {
    const float v = x[i];
    part += fmaxf(v, 0.f) - v * t + log1pf(__expf(-fabsf(v)));
    if (dx) {
      const float s = 1.f / (1.f + __expf(-v));
      dx[i * ld_dx] = __float2bfloat16(grad_scale * (s - t));
    }
  }
  part = warp_sum(part);
  __shared__ float red[32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) red[wid] = part;
  __syncthreads();
  if (wid == 0) {
    float v = lane < (blockDim.x >> 5) ? red[lane] : 0.f;
    v = warp_sum(v);
    if (lane == 0) atomicAdd(loss_acc, static_cast<double>(v));
  }
}

// ------------------------------------------------------------------------------------------------
// BatchNorm2d training-mode bookkeeping (models.py:179,181,231,239): from the fp64 sums the conv
// epilogue accumulated, produce the fused scale/shift, the saved mean / inv-std for backward, and
// update running_mean / running_var (momentum 0.1, unbiased variance) and num_batches_tracked.
// `repeat` applies the running update that many times (an elided identical forward pass, e.g. the
// reference's second generator forward, train_gan.py:56 vs 65).  The sums are re-zeroed.
// ------------------------------------------------------------------------------------------------
__global__ void bn_finalize_kernel(double* __restrict__ stats, int c, double count,
                                   const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                                   float momentum, int repeat, float* __restrict__ running_mean,
                                   float* __restrict__ running_var, long long* __restrict__ nbt,
                                   float* __restrict__ scale, float* __restrict__ shift,
                                   float* __restrict__ save_mean, float* __restrict__ save_invstd) {
  pdl_trigger();
  pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < c) {
    const double mean = stats[i] / count;
    double var = stats[c + i] / count - mean * mean;
    if (var < 0.0) var = 0.0;
    const float invstd = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
    const float g = gamma ? gamma[i] : 1.f, b = beta ? beta[i] : 0.f;
    const float sc = g * invstd;
    scale[i] = sc;
    shift[i] = b - static_cast<float>(mean) * sc;
    if (save_mean) save_mean[i] = static_cast<float>(mean);
    if (save_invstd) save_invstd[i] = invstd;
    if (running_mean) {
      const float unbiased = static_cast<float>(count > 1.0 ? var * count / (count - 1.0) : var);
      float rm = running_mean[i], rv = running_var[i];
      for (int r = 0; r < repeat; ++r) {
        rm = (1.f - momentum) * rm + momentum * static_cast<float>(mean);
        rv = (1.f - momentum) * rv + momentum * unbiased;
      }
      running_mean[i] = rm;
      running_var[i] = rv;
    }
    stats[i] = 0.0;
    stats[c + i] = 0.0;
  }
  if (i == 0 && nbt) *nbt += repeat;
}

// eval-mode scale/shift from the running statistics
__global__ void bn_eval_scale_shift_kernel(int c, const float* __restrict__ gamma, const float* __restrict__ beta,
                                           const float* __restrict__ rm, const float* __restrict__ rv, float eps,
                                           float* __restrict__ scale, float* __restrict__ shift) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < c) {
    const float sc = gamma[i] * rsqrtf(rv[i] + eps);
    scale[i] = sc;
    shift[i] = beta[i] - rm[i] * sc;
  }
}

// out1 = act1(y*scale + shift), out2 = act2(same) (optional) — 8 channels (16 bytes) per thread.
__global__ void bn_act_kernel(const __nv_bfloat16* __restrict__ y, long long ld_y, const float* __restrict__ scale,
                              const float* __restrict__ shift, long long pixels, int c,
                              __nv_bfloat16* __restrict__ o1, long long ld1, int act1,
                              __nv_bfloat16* __restrict__ o2, long long ld2, int act2) {
  pdl_trigger();
  pdl_wait();
  const int cv = c >> 3;
  const long long total = pixels * cv;
  const long long stride = (long long)gridDim.x * blockDim.x;
  constexpr int U = 4;   // independent 16-byte loads in flight per thread (the kernel is HBM-latency bound otherwise)
  for (long long i0 = blockIdx.x * (long long)blockDim.x + threadIdx.x; i0 < total; i0 += U * stride) {
    uint4 raw[U];
    long long pixv[U];
    int c8v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long i = i0 + u * stride;
      pixv[u] = i / cv;
      c8v[u] = static_cast<int>(i - pixv[u] * cv) << 3;
      if (i < total) raw[u] = __ldg(reinterpret_cast<const uint4*>(y + pixv[u] * ld_y + c8v[u]));
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (i0 + u * stride >= total) break;
      const long long pix = pixv[u];
      const int c8 = c8v[u];
      const uint32_t w[4] = {raw[u].x, raw[u].y, raw[u].z, raw[u].w};
      float v[8];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        v[2 * j] = bf16_lo(w[j]);
        v[2 * j + 1] = bf16_hi(w[j]);
      }
      const float4 s0 = *reinterpret_cast<const float4*>(scale + c8), s1 = *reinterpret_cast<const float4*>(scale + c8 + 4);
      const float4 h0 = *reinterpret_cast<const float4*>(shift + c8), h1 = *reinterpret_cast<const float4*>(shift + c8 + 4);
      const float sc[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
      const float sh[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = fmaf(v[j], sc[j], sh[j]);
      uint32_t pk[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) pk[j] = pack_bf16x2(act_fwd(v[2 * j], act1), act_fwd(v[2 * j + 1], act1));
      *reinterpret_cast<uint4*>(o1 + pix * ld1 + c8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
      if (o2) {
#pragma unroll
        for (int j = 0; j < 4; ++j) pk[j] = pack_bf16x2(act_fwd(v[2 * j], act2), act_fwd(v[2 * j + 1], act2));
        *reinterpret_cast<uint4*>(o2 + pix * ld2 + c8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// BatchNorm + activation backward.
//   yhat = y*scale + shift;  xhat = (y - mean) * invstd
//   dyhat = yhat > 0 ? (g1 + g2) : slope * g1           (g2 optional: the ReLU'd skip consumer)
//   pass 1: sums[c] += dyhat, sums[C+c] += dyhat * xhat                         (fp64 atomics)
//   pass 2: dy = scale * (dyhat - sums[c]/cnt - xhat * sums[C+c]/cnt)           (bf16)
// identity mode (scale == NULL): yhat = y, dy = dyhat (activation-only layers).
// Thread layout: threadIdx.x walks 8-channel groups, threadIdx.y walks pixels.
// ------------------------------------------------------------------------------------------------
struct BnBwdArgs {
  const __nv_bfloat16* y;
  long long ld_y;
  const __nv_bfloat16* g1;
  long long ld_g1;
  const __nv_bfloat16* g2;
  long long ld_g2;
  float slope;
  const float* scale;
  const float* shift;
  const float* mean;
  const float* invstd;
  long long pixels;
  int c;
  double* sums;
  double inv_count;
  __nv_bfloat16* dy;
  long long ld_dy;
};

__device__ __forceinline__ void load8(const __nv_bfloat16* p, float (&v)[8]) {
  const uint4 raw = *reinterpret_cast<const uint4*>(p);
  const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    v[2 * j] = bf16_lo(w[j]);
    v[2 * j + 1] = bf16_hi(w[j]);
  }
}
__device__ __forceinline__ void unpack_u4(const uint4& raw, float (&v)[8]) {
  const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    v[2 * j] = bf16_lo(w[j]);
    v[2 * j + 1] = bf16_hi(w[j]);
  }
}
__device__ __forceinline__ void loadf8(const float* p, float (&v)[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

// bn_act for the activations of the training path (identity / LeakyReLU(0.2) / ReLU), in bn_bwd_kernel's thread layout:
// threadIdx.x walks 8-channel groups, whose scale / shift stay in registers, threadIdx.y walks pixels, U pixels in
// flight per thread.  The general kernel above pays a 64-bit division, four parameter loads and a per-element
// activation switch (Tanh / Sigmoid included) per 16-byte vector: ~3500 SASS instructions, instruction-bound at
// 3.2-4.3 TB/s on the 33-134 MB tensors of the step.
__device__ __forceinline__ void act8_slope(const float (&v)[8], int act, uint32_t (&pk)[4]) {
  if (act == GAP_ACT_RELU) {
#pragma unroll
    for (int j = 0; j < 4; ++j) pk[j] = pack_bf16x2(fmaxf(v[2 * j], 0.f), fmaxf(v[2 * j + 1], 0.f));
  } else if (act == GAP_ACT_LRELU) {      // v > 0 ? v : 0.2 v  ==  max(v, 0.2 v)
#pragma unroll
    for (int j = 0; j < 4; ++j) pk[j] = pack_bf16x2(fmaxf(v[2 * j], 0.2f * v[2 * j]), fmaxf(v[2 * j + 1], 0.2f * v[2 * j + 1]));
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) pk[j] = pack_bf16x2(v[2 * j], v[2 * j + 1]);
  }
}

template <int U>
__global__ void __launch_bounds__(256, 3) bn_act_slope_kernel(const __nv_bfloat16* __restrict__ y, long long ld_y,
                                                           const float* __restrict__ scale, const float* __restrict__ shift,
                                                           long long pixels, int c, __nv_bfloat16* __restrict__ o1,
                                                           long long ld1, int act1, __nv_bfloat16* __restrict__ o2,
                                                           long long ld2, int act2) {
  pdl_trigger();
  pdl_wait();
  const int cv = c >> 3;
  const long long pstride = (long long)gridDim.x * blockDim.y;
  for (int cg = threadIdx.x; cg < cv; cg += blockDim.x) {
    const int c8 = cg << 3;
    float sc[8], sh[8];
    loadf8(scale + c8, sc);
    loadf8(shift + c8, sh);
    for (long long pix0 = blockIdx.x * (long long)blockDim.y + threadIdx.y; pix0 < pixels; pix0 += U * pstride) {
      uint4 raw[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long pix = pix0 + u * pstride;
        if (pix < pixels) raw[u] = __ldg(reinterpret_cast<const uint4*>(y + pix * ld_y + c8));
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long pix = pix0 + u * pstride;
        if (pix >= pixels) break;
        float v[8];
        unpack_u4(raw[u], v);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = fmaf(v[j], sc[j], sh[j]);
        uint32_t pk[4];
        act8_slope(v, act1, pk);
        *reinterpret_cast<uint4*>(o1 + pix * ld1 + c8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        if (o2) {
          act8_slope(v, act2, pk);
          *reinterpret_cast<uint4*>(o2 + pix * ld2 + c8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
      }
    }
  }
}

// G2: a second gradient source exists (its registers disappear otherwise); U: pixels in flight per thread (six instead
// of four measured no gain: 65.6 -> 68.3, 37.6 -> 36.4, 19.2 -> 19.2, 35.5 -> 34.8 us, tools/bench_bn_act.py).
template <bool APPLY, bool G2, int U>
__global__ void __launch_bounds__(256, 2) bn_bwd_kernel(const BnBwdArgs a) {
  pdl_trigger();
  pdl_wait();
  const int cv = a.c >> 3;
  const bool ident = a.scale == nullptr;
  extern __shared__ float sm_red[];  // [blockDim.y][cv*8][2] for the reduce pass
  for (int cg = threadIdx.x; cg < cv; cg += blockDim.x) {
    const int c8 = cg << 3;
    // per-channel constants, folded so that few registers stay live:
    //   mask:   y*sc + sh > 0
    //   apply:  dy = sc*(d - m1 - xhat*m2) = sc*d + ca*y + cb,  ca = -sc*m2*invstd, cb = -sc*m1 - ca*mean
    //   reduce: sums of d and d*y (converted to sum d*xhat = invstd*(sum d*y - mean*sum d) at the end)
    float sc[8], sh[8], ca[8], cb[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      sc[j] = ident ? 1.f : a.scale[c8 + j];
      sh[j] = ident ? 0.f : a.shift[c8 + j];
      ca[j] = 0.f;
      cb[j] = 0.f;
    }
    if (APPLY && !ident) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const double t1 = a.sums[c8 + j];
        const double t2 = a.sums[a.c + c8 + j];
        const float m1 = static_cast<float>(t1 * a.inv_count);
        const float m2 = static_cast<float>(t2 * a.inv_count);
        ca[j] = -sc[j] * m2 * a.invstd[c8 + j];
        cb[j] = -sc[j] * m1 - ca[j] * a.mean[c8 + j];
      }
    }
    float s1[8] = {0, 0, 0, 0, 0, 0, 0, 0}, s2[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    // pixels in flight per thread: loads of all U issued before any use
    const long long pstride = (long long)gridDim.x * blockDim.y;
    for (long long pix0 = blockIdx.x * (long long)blockDim.y + threadIdx.y; pix0 < a.pixels; pix0 += U * pstride) {
      uint4 yr[U], g1r[U], g2r[G2 ? U : 1];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long pix = pix0 + u * pstride;
        if (pix < a.pixels) {
          yr[u] = __ldg(reinterpret_cast<const uint4*>(a.y + pix * a.ld_y + c8));
          g1r[u] = __ldg(reinterpret_cast<const uint4*>(a.g1 + pix * a.ld_g1 + c8));
          if (G2) g2r[u] = __ldg(reinterpret_cast<const uint4*>(a.g2 + pix * a.ld_g2 + c8));
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long pix = pix0 + u * pstride;
        if (pix >= a.pixels) break;
        float y[8], g1[8], g2[8];
        unpack_u4(yr[u], y);
        unpack_u4(g1r[u], g1);
        if (G2) unpack_u4(g2r[G2 ? u : 0], g2);
        float d[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float yh = fmaf(y[j], sc[j], sh[j]);
          const float gp = G2 ? g1[j] + g2[j] : g1[j];
          d[j] = yh > 0.f ? gp : a.slope * g1[j];
        }
        if (APPLY) {
          uint32_t pk[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            float o0 = d[2 * j], o1 = d[2 * j + 1];
            if (!ident) {
              o0 = fmaf(sc[2 * j], o0, fmaf(ca[2 * j], y[2 * j], cb[2 * j]));
              o1 = fmaf(sc[2 * j + 1], o1, fmaf(ca[2 * j + 1], y[2 * j + 1], cb[2 * j + 1]));
            }
            pk[j] = pack_bf16x2(o0, o1);
          }
          *reinterpret_cast<uint4*>(a.dy + pix * a.ld_dy + c8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            s1[j] += d[j];
            s2[j] += d[j] * y[j];
          }
        }
      }
    }
    if (!APPLY) {
      float* slot = sm_red + (static_cast<size_t>(threadIdx.y) * cv * 8 + c8) * 2;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        // sum d*xhat = invstd * (sum d*y - mean * sum d)
        const float mu = ident ? 0.f : a.mean[c8 + j], is = ident ? 0.f : a.invstd[c8 + j];
        slot[2 * j] = s1[j];
        slot[2 * j + 1] = is * (s2[j] - mu * s1[j]);
      }
    }
  }
  if (!APPLY) {
    __syncthreads();
    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    const int nthr = blockDim.x * blockDim.y;
    for (int i = tid; i < a.c * 2; i += nthr) {
      const int ch = i >> 1, which = i & 1;
      double tot = 0.0;
      for (int r = 0; r < blockDim.y; ++r) tot += sm_red[(static_cast<size_t>(r) * cv * 8 + ch) * 2 + which];
      atomicAdd(a.sums + which * a.c + ch, tot);
    }
  }
}

// dgamma = sums[C+c], dbeta = sums[c] (accumulated into fp32 grads), then re-zero the sums.
__global__ void bn_param_grads_kernel(double* __restrict__ sums, int c, float* __restrict__ dgamma,
                                      float* __restrict__ dbeta) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < c) {
    if (dbeta) dbeta[i] += static_cast<float>(sums[i]);
    if (dgamma) dgamma[i] += static_cast<float>(sums[c + i]);
    sums[i] = 0.0;
    sums[c + i] = 0.0;
  }
}

// raw = [sum d, sum d*y] from the backward-fused GEMM epilogue -> sums = [sum d, sum d*xhat]; parameter
// gradients; raw re-zeroed for the next backward pass.
__global__ void bn_bwd_finalize_kernel(double* __restrict__ raw, const float* __restrict__ mean,
                                       const float* __restrict__ invstd, int c, float* __restrict__ dgamma,
                                       float* __restrict__ dbeta, double* __restrict__ sums) {
  pdl_trigger();
  pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < c) {
    const double s1 = raw[i], s2 = raw[c + i];
    const double sx = static_cast<double>(invstd[i]) * (s2 - static_cast<double>(mean[i]) * s1);
    sums[i] = s1;
    sums[c + i] = sx;
    if (dbeta) dbeta[i] += static_cast<float>(s1);
    if (dgamma) dgamma[i] += static_cast<float>(sx);
    raw[i] = 0.0;
    raw[c + i] = 0.0;
  }
}

// per-channel column sums of a bf16 [pixels][c] tensor into fp32 (bias gradients)
__global__ void colsum_kernel(const __nv_bfloat16* __restrict__ x, long long ld, long long pixels, int c,
                              float* __restrict__ out) {
  // 256 threads = (256/cpad) pixel lanes x cpad channel lanes, cpad = pow2 >= min(c, 256)
  __shared__ float red[256];
  int cpad = 1;
  while (cpad < c && cpad < 256) cpad <<= 1;
  const int lanes = 256 / cpad;
  const int cl = threadIdx.x % cpad, pl = threadIdx.x / cpad;
  for (int ch = cl; ch < c; ch += cpad) {
    float s = 0.f;
    for (long long pix = static_cast<long long>(blockIdx.x) * lanes + pl; pix < pixels;
         pix += static_cast<long long>(gridDim.x) * lanes)
      s += __bfloat162float(x[pix * ld + ch]);
    red[threadIdx.x] = s;
    __syncthreads();
    if (pl == 0) {
      for (int r = 1; r < lanes; ++r) s += red[r * cpad + cl];
      atomicAdd(out + ch, s);
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// Adam / AdamW on a flat fp32 buffer (torch.optim semantics; train_gan.py:140-141, train.py:295)
// ------------------------------------------------------------------------------------------------
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, long long n, float lr, float b1, float b2, float eps,
                            float wd, int decoupled, float bc1, float bc2_sqrt, float grad_scale,
                            const int* __restrict__ step_dev) {
  const long long n4 = n >> 2;
  if (step_dev != nullptr) {
    // step counter kept on the device (CUDA-graph replay): bias corrections computed here
    const double st = static_cast<double>(*step_dev);
    bc1 = static_cast<float>(1.0 - pow(static_cast<double>(b1), st));
    bc2_sqrt = static_cast<float>(sqrt(1.0 - pow(static_cast<double>(b2), st)));
  }
  const float step_size = lr / bc1;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4;
       i += (long long)gridDim.x * blockDim.x) {
    float4 pp = reinterpret_cast<float4*>(p)[i];
    const float4 gg = reinterpret_cast<const float4*>(g)[i];
    float4 mm = reinterpret_cast<float4*>(m)[i];
    float4 vv = reinterpret_cast<float4*>(v)[i];
    float* pa = &pp.x;
    const float* ga = &gg.x;
    float* ma = &mm.x;
    float* va = &vv.x;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float gr = ga[j] * grad_scale;
      if (decoupled) pa[j] *= (1.f - lr * wd);
      else if (wd != 0.f) gr += wd * pa[j];
      ma[j] = b1 * ma[j] + (1.f - b1) * gr;
      va[j] = b2 * va[j] + (1.f - b2) * gr * gr;
      const float denom = sqrtf(va[j]) / bc2_sqrt + eps;
      pa[j] -= step_size * (ma[j] / denom);
    }
    reinterpret_cast<float4*>(p)[i] = pp;
    reinterpret_cast<float4*>(m)[i] = mm;
    reinterpret_cast<float4*>(v)[i] = vv;
  }
  // tail
  const long long tail0 = n4 << 2;
  for (long long i = tail0 + blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x) {
    float gr = g[i] * grad_scale;
    float pv = p[i];
    if (decoupled) pv *= (1.f - lr * wd);
    else if (wd != 0.f) gr += wd * pv;
    const float mv = b1 * m[i] + (1.f - b1) * gr;
    const float vv2 = b2 * v[i] + (1.f - b2) * gr * gr;
    m[i] = mv;
    v[i] = vv2;
    p[i] = pv - step_size * (mv / (sqrtf(vv2) / bc2_sqrt + eps));
  }
}

// ------------------------------------------------------------------------------------------------
// Weight packing: fp32 master weights (any strides) -> bf16 K-major GEMM operand
//   out[p][r][t*c_pad + c] = w[r*s_r + c*s_c + kh*s_kh + kw*s_kw]   (zero where c >= C, r >= R,
//   or beyond taps*c_pad), (kh,kw) from (phase p, tap t) by `mode`:
//   0 direct (kh=th,kw=tw)   1 flipped (kh=KH-1-th)   2 k4s2p1 phases (kh=3-ph-2th, kw=3-pw-2tw)
// mode 3 ("col-T"): rows are (tap, c) pairs: out[0][t*C + c][k] = w[k*s_r + c*s_c + kh*s_kh + kw*s_kw]
// ------------------------------------------------------------------------------------------------
struct PackArgs {
  const float* w;
  __nv_bfloat16* out;
  int mode, n_phase, rows, rows_pad, taps_h, taps_w, c, c_pad, krow;
  long long s_r, s_c, s_kh, s_kw;
  int kdim;  // mode 3: valid K (source "row" count)
};

__global__ void pack_weights_kernel(const PackArgs a) {
  const long long total = static_cast<long long>(a.n_phase) * a.rows_pad * a.krow;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int k = static_cast<int>(i % a.krow);
    const int r = static_cast<int>((i / a.krow) % a.rows_pad);
    const int p = static_cast<int>(i / (static_cast<long long>(a.krow) * a.rows_pad));
    float v = 0.f;
    if (a.mode == 3) {
      const int t = r / a.c, c = r - t * a.c;
      if (r < a.rows && k < a.kdim) {
        const int kh = t / a.taps_w, kw = t - kh * a.taps_w;
        v = a.w[k * a.s_r + c * a.s_c + kh * a.s_kh + kw * a.s_kw];
      }
    } else {
      const int t = k / a.c_pad, c = k - t * a.c_pad;
      if (r < a.rows && t < a.taps_h * a.taps_w && c < a.c) {
        const int th = t / a.taps_w, tw = t - th * a.taps_w;
        int kh = th, kw = tw;
        if (a.mode == 1) {
          kh = a.taps_h - 1 - th;
          kw = a.taps_w - 1 - tw;
        } else if (a.mode == 2) {
          kh = 3 - (p >> 1) - 2 * th;
          kw = 3 - (p & 1) - 2 * tw;
        }
        v = a.w[r * a.s_r + c * a.s_c + kh * a.s_kh + kw * a.s_kw];
      }
    }
    a.out[i] = __float2bfloat16(v);
  }
}


// ------------------------------------------------------------------------------------------------
// Multi-tensor weight packing: every fp32 master -> bf16 GEMM operand of a network in ONE launch.
// One CTA = one 32 x 32 (row, channel) tile of one (phase, tap) slice of one table entry; reads run
// along whichever of (row, channel) is contiguous in the master, writes along the channel (K) axis
// of the operand, through a padded shared-memory tile when the two differ.  Padding elements of the
// operand are never written: the caller zero-fills the operand buffers once.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pack_weights_multi_kernel(const gap_pack_entry* __restrict__ table,
                                                                 int n_entries) {
  // One CTA = one 64 x 64 (row, channel) tile of one (phase, tap) slice of one table entry.
  __shared__ float tile[64][65];
  __shared__ int s_entry;
  if (threadIdx.x == 0 && threadIdx.y == 0) {
    int lo = 0, hi = n_entries - 1;   // last entry whose tile_begin <= blockIdx.x
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (table[mid].tile_begin <= static_cast<int>(blockIdx.x)) lo = mid;
      else hi = mid - 1;
    }
    s_entry = lo;
  }
  __syncthreads();
  const gap_pack_entry a = table[s_entry];
  int t = blockIdx.x - a.tile_begin;
  const int tc = t % a.tiles_c;
  t /= a.tiles_c;
  const int tr = t % a.tiles_r;
  t /= a.tiles_r;
  const int n_taps = a.taps_h * a.taps_w;
  const int tap = t % n_taps;
  const int ph = t / n_taps;
  const int th = tap / a.taps_w, tw = tap - th * a.taps_w;
  int kh = th, kw = tw;
  if (a.mode == 1) {
    kh = a.taps_h - 1 - th;
    kw = a.taps_w - 1 - tw;
  } else if (a.mode == 2) {
    kh = 3 - (ph >> 1) - 2 * th;
    kw = 3 - (ph & 1) - 2 * tw;
  }
  const float* __restrict__ w = a.w + kh * a.s_kh + kw * a.s_kw;
  __nv_bfloat16* __restrict__ out = static_cast<__nv_bfloat16*>(a.out) +
                                    static_cast<long long>(ph) * a.rows_pad * a.krow + tap * a.c_pad;
  const int r0 = tr * 64, c0 = tc * 64;
  const int tid = threadIdx.y * 32 + threadIdx.x;
  const int tx16 = tid & 15, ty16 = tid >> 4;     // 16 x 16 thread layout: 4 elements along the fast axis each
  const bool out_vec = (a.krow % 4 == 0) && (a.c_pad % 4 == 0) && ((reinterpret_cast<uintptr_t>(a.out) & 7) == 0);
  if (a.s_r == 1 && a.s_c != 1) {
    // master contiguous along rows: read float4 along r, transpose through shared memory, write along c
    const bool in_vec = (a.s_c % 4 == 0) && (a.s_kh % 4 == 0) && (a.s_kw % 4 == 0) &&
                        ((reinterpret_cast<uintptr_t>(a.w) & 15) == 0);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int c = c0 + ty16 + 16 * i, r = r0 + tx16 * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c < a.c) {
        const float* src = w + r + static_cast<long long>(c) * a.s_c;
        if (in_vec && r + 3 < a.rows) {
          v = __ldg(reinterpret_cast<const float4*>(src));
        } else {
          if (r < a.rows) v.x = src[0];
          if (r + 1 < a.rows) v.y = src[1];
          if (r + 2 < a.rows) v.z = src[2];
          if (r + 3 < a.rows) v.w = src[3];
        }
      }
      tile[ty16 + 16 * i][tx16 * 4 + 0] = v.x;
      tile[ty16 + 16 * i][tx16 * 4 + 1] = v.y;
      tile[ty16 + 16 * i][tx16 * 4 + 2] = v.z;
      tile[ty16 + 16 * i][tx16 * 4 + 3] = v.w;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = r0 + ty16 + 16 * i, c = c0 + tx16 * 4;
      if (r >= a.rows || c >= a.c) continue;
      __nv_bfloat16* dst = out + static_cast<long long>(r) * a.krow + c;
      const float v0 = tile[tx16 * 4 + 0][ty16 + 16 * i], v1 = tile[tx16 * 4 + 1][ty16 + 16 * i];
      const float v2 = tile[tx16 * 4 + 2][ty16 + 16 * i], v3 = tile[tx16 * 4 + 3][ty16 + 16 * i];
      if (out_vec && c + 3 < a.c) {
        *reinterpret_cast<uint2*>(dst) = make_uint2(pack_bf16x2(v0, v1), pack_bf16x2(v2, v3));
      } else {
        dst[0] = __float2bfloat16(v0);
        if (c + 1 < a.c) dst[1] = __float2bfloat16(v1);
        if (c + 2 < a.c) dst[2] = __float2bfloat16(v2);
        if (c + 3 < a.c) dst[3] = __float2bfloat16(v3);
      }
    }
  } else {
    const bool in_vec = (a.s_c == 1) && (a.s_r % 4 == 0) && (a.s_kh % 4 == 0) && (a.s_kw % 4 == 0) &&
                        ((reinterpret_cast<uintptr_t>(a.w) & 15) == 0);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = r0 + ty16 + 16 * i, c = c0 + tx16 * 4;
      if (r >= a.rows || c >= a.c) continue;
      const float* src = w + static_cast<long long>(r) * a.s_r + static_cast<long long>(c) * a.s_c;
      float v0, v1 = 0.f, v2 = 0.f, v3 = 0.f;
      if (in_vec && c + 3 < a.c) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(src));
        v0 = v.x; v1 = v.y; v2 = v.z; v3 = v.w;
      } else {
        v0 = src[0];
        if (c + 1 < a.c) v1 = src[a.s_c];
        if (c + 2 < a.c) v2 = src[2 * a.s_c];
        if (c + 3 < a.c) v3 = src[3 * a.s_c];
      }
      __nv_bfloat16* dst = out + static_cast<long long>(r) * a.krow + c;
      if (out_vec && c + 3 < a.c) {
        *reinterpret_cast<uint2*>(dst) = make_uint2(pack_bf16x2(v0, v1), pack_bf16x2(v2, v3));
      } else {
        dst[0] = __float2bfloat16(v0);
        if (c + 1 < a.c) dst[1] = __float2bfloat16(v1);
        if (c + 2 < a.c) dst[2] = __float2bfloat16(v2);
        if (c + 3 < a.c) dst[3] = __float2bfloat16(v3);
      }
    }
  }
}

}  // namespace gap

using namespace gap;

#define GAP_LAUNCH_CHECK()                 \
  do {                                     \
    GAP_CUDA(cudaGetLastError());          \
  } while (0)

extern "C" {

int gap_nchw_f32_to_nhwc_bf16(const float* x, void* out, int n, int c, int h, int w, int64_t out_ld,
                              void* stream) {
  GAP_CHECK_ARG(x && out && n > 0 && c > 0 && c <= out_ld, "gap_nchw_f32_to_nhwc_bf16: bad arguments");
  const long long hw = static_cast<long long>(h) * w;
  if (c <= 4 && out_ld == 4 && hw % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
      (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
    // (slots >= c are written as zero, which is what the 4-slot image layout holds there anyway)
    const long long total4 = n * hw / 4;
    const int grid = grid_even(total4, 256, 148 * 8);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    __nv_bfloat16* o = static_cast<__nv_bfloat16*>(out);
    switch (c) {
      case 1: nchw_f32_to_nhwc4_bf16_kernel<1><<<grid, 256, 0, st>>>(x, o, hw / 4, total4); break;
      case 2: nchw_f32_to_nhwc4_bf16_kernel<2><<<grid, 256, 0, st>>>(x, o, hw / 4, total4); break;
      case 3: nchw_f32_to_nhwc4_bf16_kernel<3><<<grid, 256, 0, st>>>(x, o, hw / 4, total4); break;
      default: nchw_f32_to_nhwc4_bf16_kernel<4><<<grid, 256, 0, st>>>(x, o, hw / 4, total4); break;
    }
    GAP_LAUNCH_CHECK();
    return 0;
  }
  nchw_f32_to_nhwc_bf16_kernel<<<grid_for(n * hw, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      x, static_cast<__nv_bfloat16*>(out), n, c, hw, out_ld);
  GAP_LAUNCH_CHECK();
  return 0;
}

int gap_nhwc_to_nchw_f32(const void* x, int x_is_f32, float* out, int n, int c, int h, int w, int64_t x_ld,
                         int c_total, int c_off, void* stream) {
  GAP_CHECK_ARG(x && out && n > 0 && c > 0 && c <= x_ld && c_off >= 0 && c_off + c <= c_total,
                "gap_nhwc_to_nchw_f32: bad arguments");
  const long long hw = static_cast<long long>(h) * w;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (x_is_f32)
    nhwc_to_nchw_f32_kernel<float><<<grid_for(n * hw, 256), 256, 0, st>>>(static_cast<const float*>(x), out, n, c, hw,
                                                                          x_ld, c_total, c_off);
  else
    nhwc_to_nchw_f32_kernel<__nv_bfloat16><<<grid_for(n * hw, 256), 256, 0, st>>>(
        static_cast<const __nv_bfloat16*>(x), out, n, c, hw, x_ld, c_total, c_off);
  GAP_LAUNCH_CHECK();
  return 0;
}

int gap_tanh_bwd(const float* gout_nchw, const float* y_nhwc, int64_t ld_y, void* dpre, int64_t ld_p, int n, int c,
                 int h, int w, void* stream) {
  GAP_CHECK_ARG(gout_nchw && y_nhwc && dpre && n > 0 && c > 0, "gap_tanh_bwd: bad arguments");
  const long long hw = static_cast<long long>(h) * w;
  tanh_bwd_kernel<<<grid_for(n * hw, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      gout_nchw, y_nhwc, ld_y, static_cast<__nv_bfloat16*>(dpre), ld_p, n, c, hw);
  GAP_LAUNCH_CHECK();
  return 0;
}

// the four-pixel kernel: 1..4 channels in dense 4-slot tensors, whole quads inside one image, 16-byte aligned pointers
static bool gen_out_vec_ok(const void* fake, const void* real, const void* dfake_d, const void* dpre, int64_t ld_f,
                           int64_t ld_d, int64_t ld_p, int64_t hw, int c) {
  if (debug_get("gen_out_c3", 1) == 0) return false;
  auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  return c <= 4 && ld_f == 4 && ld_p == 4 && (!dfake_d || ld_d == 4) && hw % 4 == 0 && al16(fake) && al16(real) &&
         al16(dfake_d) && al16(dpre);
}

int gap_gen_out_bwd(const float* fake, int64_t ld_f, const float* real_nchw, int64_t hw, const float* dfake_d,
                    int64_t ld_d, float l1_scale, void* dpre, int64_t ld_p, int64_t pixels, int c,
                    double* loss_acc, void* stream) {
  GAP_CHECK_ARG(fake && real_nchw && dpre && loss_acc && pixels > 0 && c > 0 && hw > 0 && pixels % hw == 0,
                "gap_gen_out_bwd: bad arguments");
  if (gen_out_vec_ok(fake, real_nchw, dfake_d, dpre, ld_f, ld_d, ld_p, hw, c)) {
    gen_out_bwd_vec_launch<false>(fake, real_nchw, hw, dfake_d, l1_scale, dpre, pixels, c, loss_acc,
                                  static_cast<cudaStream_t>(stream));
    GAP_LAUNCH_CHECK();
    return 0;
  }
  gen_out_bwd_kernel<false><<<grid_for(pixels, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      fake, ld_f, real_nchw, hw, dfake_d, ld_d, l1_scale, static_cast<__nv_bfloat16*>(dpre), ld_p, pixels, c,
      loss_acc);
  GAP_LAUNCH_CHECK();
  return 0;
}

int gap_gen_out_bwd_u8(const float* fake, int64_t ld_f, const uint8_t* real_hwc, int64_t hw, const float* dfake_d,
                       int64_t ld_d, float l1_scale, void* dpre, int64_t ld_p, int64_t pixels, int c,
                       double* loss_acc, void* stream) {
  GAP_CHECK_ARG(fake && real_hwc && dpre && loss_acc && pixels > 0 && c > 0 && hw > 0 && pixels % hw == 0,
                "gap_gen_out_bwd_u8: bad arguments");
  if (gen_out_vec_ok(fake, real_hwc, dfake_d, dpre, ld_f, ld_d, ld_p, hw, c) && (reinterpret_cast<uintptr_t>(real_hwc) & 3) == 0) {
    gen_out_bwd_vec_launch<true>(fake, real_hwc, hw, dfake_d, l1_scale, dpre, pixels, c, loss_acc,
                                 static_cast<cudaStream_t>(stream));
    GAP_LAUNCH_CHECK();
    return 0;
  }
  gen_out_bwd_kernel<true><<<grid_for(pixels, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      fake, ld_f, real_hwc, hw, dfake_d, ld_d, l1_scale, static_cast<__nv_bfloat16*>(dpre), ld_p, pixels, c, loss_acc);
  GAP_LAUNCH_CHECK();
  return 0;
}

int gap_bce_logits_const(const float* logits, int64_t count, float target, float grad_scale, void* dlogits,
                         int64_t ld_d, double* loss_acc, void* stream) {
  GAP_CHECK_ARG(logits && loss_acc && count > 0, "gap_bce_logits_const: bad arguments");
  bce_logits_const_kernel<<<grid_for(count, 256, 148), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      logits, count, target, grad_scale, static_cast<__nv_bfloat16*>(dlogits), ld_d, loss_acc);
  GAP_LAUNCH_CHECK();
  return 0;
}

int gap_bn_finalize(double* stats, int c, double count, const float* gamma, const float* beta, float eps,
                    float momentum, int repeat, float* running_mean, float* running_var, int64_t* nbt,
                    float* scale, float* shift, float* save_mean, float* save_invstd, void* stream) {
  GAP_CHECK_ARG(stats && scale && shift && c > 0 && count > 0, "gap_bn_finalize: bad arguments");
  GAP_CUDA(launch_pdl(bn_finalize_kernel, dim3((c + 127) / 128), dim3(128), 0, static_cast<cudaStream_t>(stream), stats, c,
                      count, gamma, beta, eps, momentum, repeat, running_mean, running_var,
                      reinterpret_cast<long long*>(nbt), scale, shift, save_mean, save_invstd));
  GAP_LAUNCH_CHECK();
  return 0;
}

int gap_bn_eval_scale_shift(int c, const float* gamma, const float* beta, const float* running_mean,
                            const float* running_var, float eps, float* scale, float* shift, void* stream) {
  GAP_CHECK_ARG(gamma && beta && running_mean && running_var && scale && shift && c > 0,
                "gap_bn_eval_scale_shift: bad arguments");
  bn_eval_scale_shift_kernel<<<(c + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      c, gamma, beta, running_mean, running_var, eps, scale, shift);
  GAP_LAUNCH_CHECK();
  return 0;
}

int gap_bn_act(const void* y, int64_t ld_y, const float* scale, const float* shift, int64_t pixels, int c,
               void* out1, int64_t ld1, int act1, void* out2, int64_t ld2, int act2, void* stream) {
  GAP_CHECK_ARG(y && scale && shift && out1 && pixels > 0 && c > 0 && c % 8 == 0, "gap_bn_act: bad arguments");
  if (ld_y % 8 || ld1 % 8 || (out2 && ld2 % 8)) {
    set_error("gap_bn_act: pixel strides must be multiples of 8");
    return GAP_ERR_ALIGNMENT;
  }
  auto slope_type = [](int a) { return a == GAP_ACT_NONE || a == GAP_ACT_LRELU || a == GAP_ACT_RELU; };
  if (slope_type(act1) && (!out2 || slope_type(act2)) && debug_get("bn_act_fast", 1) != 0) {
    const int cv = c / 8;
    const int bx = cv < 128 ? cv : 128;
    const int by = 256 / bx < 1 ? 1 : 256 / bx;
    const long long slabs = (pixels + by - 1) / by;
    // three resident blocks per SM (78 registers): measured 45.8 / 25.9 / 13.0 us on the 128 / 64 / 32-pixel-wide
    // batch-64 tensors against 55.7 / 31.0 / 17.6 us of the general kernel (tools/bench_bn_act.py)
    GAP_CUDA(launch_pdl(bn_act_slope_kernel<4>, dim3(grid_even(slabs, 4, 148 * debug_get("bn_act_bps", 3))), dim3(bx, by), 0,
                        static_cast<cudaStream_t>(stream), static_cast<const __nv_bfloat16*>(y), static_cast<long long>(ld_y),
                        scale, shift, static_cast<long long>(pixels), c, static_cast<__nv_bfloat16*>(out1),
                        static_cast<long long>(ld1), act1, static_cast<__nv_bfloat16*>(out2), static_cast<long long>(ld2),
                        act2));
    GAP_LAUNCH_CHECK();
    return 0;
  }
  // 4 vectors per thread and sweep (U in the kernel)
  GAP_CUDA(launch_pdl(bn_act_kernel, dim3(grid_even(pixels * (c / 8), 256 * 4, 148 * debug_get("bn_act_bps", 4))), dim3(256), 0, static_cast<cudaStream_t>(stream),
                      static_cast<const __nv_bfloat16*>(y), static_cast<long long>(ld_y), scale, shift,
                      static_cast<long long>(pixels), c, static_cast<__nv_bfloat16*>(out1), static_cast<long long>(ld1),
                      act1, static_cast<__nv_bfloat16*>(out2), static_cast<long long>(ld2), act2));
  GAP_LAUNCH_CHECK();
  return 0;
}

static int bn_bwd_launch(bool apply, const BnBwdArgs& a, cudaStream_t st) {
  const int cv = a.c / 8;
  int bx = cv < 128 ? cv : 128;
  int by = 256 / bx;
  if (by < 1) by = 1;
  dim3 block(bx, by);
  const long long slabs = (a.pixels + by - 1) / by;
  const bool g2 = a.g2 != nullptr;
  const int grid = grid_even(slabs, 4, 148 * debug_get("bn_bwd_bps", 2));   // 4 pixel slabs per block and sweep (U in the kernel); resident blocks only
  if (apply) {
    if (g2)
      GAP_CUDA(launch_pdl(bn_bwd_kernel<true, true, 4>, dim3(grid), block, 0, st, a));
    else
      GAP_CUDA(launch_pdl(bn_bwd_kernel<true, false, 4>, dim3(grid), block, 0, st, a));
  } else {
    const size_t smem = static_cast<size_t>(by) * a.c * 2 * sizeof(float);
    if (smem > 48 * 1024) {
      static bool set = false;
      if (!set) {
        GAP_CUDA(cudaFuncSetAttribute(bn_bwd_kernel<false, true, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
        GAP_CUDA(cudaFuncSetAttribute(bn_bwd_kernel<false, false, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
        set = true;
      }
    }
    if (g2)
      GAP_CUDA(launch_pdl(bn_bwd_kernel<false, true, 4>, dim3(grid), block, smem, st, a));
    else
      GAP_CUDA(launch_pdl(bn_bwd_kernel<false, false, 4>, dim3(grid), block, smem, st, a));
  }
  GAP_CUDA(cudaGetLastError());
  return 0;
}

int gap_bn_bwd_reduce(const void* y, int64_t ld_y, const void* g1, int64_t ld_g1, const void* g2, int64_t ld_g2,
                      float slope, const float* scale, const float* shift, const float* mean,
                      const float* invstd, int64_t pixels, int c, double* sums, void* stream) {
  GAP_CHECK_ARG(y && g1 && scale && shift && mean && invstd && sums && pixels > 0 && c > 0 && c % 8 == 0,
                "gap_bn_bwd_reduce: bad arguments");
  BnBwdArgs a{static_cast<const __nv_bfloat16*>(y), ld_y, static_cast<const __nv_bfloat16*>(g1), ld_g1,
              static_cast<const __nv_bfloat16*>(g2), ld_g2, slope, scale, shift, mean, invstd, pixels, c, sums,
              0.0, nullptr, 0};
  return bn_bwd_launch(false, a, static_cast<cudaStream_t>(stream));
}

int gap_bn_bwd_apply(const void* y, int64_t ld_y, const void* g1, int64_t ld_g1, const void* g2, int64_t ld_g2,
                     float slope, const float* scale, const float* shift, const float* mean, const float* invstd,
                     int64_t pixels, int c, const double* sums, double count, void* dy, int64_t ld_dy,
                     void* stream) {
  GAP_CHECK_ARG(y && g1 && dy && pixels > 0 && c > 0 && c % 8 == 0, "gap_bn_bwd_apply: bad arguments");
  GAP_CHECK_ARG(scale == nullptr || (shift && mean && invstd && sums && count > 0),
                "gap_bn_bwd_apply: BatchNorm mode needs shift/mean/invstd/sums/count");
  BnBwdArgs a{static_cast<const __nv_bfloat16*>(y), ld_y, static_cast<const __nv_bfloat16*>(g1), ld_g1,
              static_cast<const __nv_bfloat16*>(g2), ld_g2, slope, scale, shift, mean, invstd, pixels, c,
              const_cast<double*>(sums), count > 0 ? 1.0 / count : 0.0, static_cast<__nv_bfloat16*>(dy), ld_dy};
  return bn_bwd_launch(true, a, static_cast<cudaStream_t>(stream));
}

int gap_bn_param_grads(double* sums, int c, float* dgamma, float* dbeta, void* stream) {
  GAP_CHECK_ARG(sums && c > 0, "gap_bn_param_grads: bad arguments");
  bn_param_grads_kernel<<<(c + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(sums, c, dgamma, dbeta);
  GAP_LAUNCH_CHECK();
  return 0;
}

int gap_bn_bwd_finalize(double* raw, const float* mean, const float* invstd, int c, float* dgamma, float* dbeta,
                        double* sums, void* stream) {
  GAP_CHECK_ARG(raw && mean && invstd && sums && c > 0, "gap_bn_bwd_finalize: bad arguments");
  GAP_CUDA(launch_pdl(bn_bwd_finalize_kernel, dim3((c + 127) / 128), dim3(128), 0, static_cast<cudaStream_t>(stream), raw,
                      mean, invstd, c, dgamma, dbeta, sums));
  GAP_LAUNCH_CHECK();
  return 0;
}

int gap_colsum_bf16(const void* x, int64_t ld, int64_t pixels, int c, float* out, void* stream) {
  GAP_CHECK_ARG(x && out && pixels > 0 && c > 0, "gap_colsum_bf16: bad arguments");
  const int block = 256;
  const int grid = static_cast<int>(pixels < 148 * 8 ? pixels : 148 * 8);
  colsum_kernel<<<grid, block, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const __nv_bfloat16*>(x), ld,
                                                                      pixels, c, out);
  GAP_LAUNCH_CHECK();
  return 0;
}

int gap_adam_flat(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                  float eps, float weight_decay, int decoupled, int step, float grad_scale, void* stream) {
  GAP_CHECK_ARG(p && g && m && v && n > 0 && step >= 1, "gap_adam_flat: bad arguments");
  if ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) |
       reinterpret_cast<uintptr_t>(v)) & 15) {
    set_error("gap_adam_flat: buffers must be 16-byte aligned");
    return GAP_ERR_ALIGNMENT;
  }
  const double bc1 = 1.0 - pow(static_cast<double>(beta1), step);
  const double bc2 = 1.0 - pow(static_cast<double>(beta2), step);
  adam_kernel<<<grid_for(n / 4 + 1, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      p, g, m, v, n, lr, beta1, beta2, eps, weight_decay, decoupled, static_cast<float>(bc1),
      static_cast<float>(sqrt(bc2)), grad_scale, nullptr);
  GAP_LAUNCH_CHECK();
  return 0;
}

// train_gan.py:61,68-69 from the four loss sums of one iteration (fp64): acc = [sum BCE(D(real),1), sum BCE(D(fake),0),
// sum BCE(D(fake),1), sum |fake - real|] -> out = [loss_D, loss_G]; acc is re-zeroed for the next iteration.
__global__ void gan_losses_kernel(double* acc, double inv_cnt, double l1_weight_over_numel, double* out) {
  if (threadIdx.x == 0) {
    out[0] = 0.5 * (acc[0] + acc[1]) * inv_cnt;
    out[1] = acc[2] * inv_cnt + l1_weight_over_numel * acc[3];
    acc[0] = acc[1] = acc[2] = acc[3] = 0.0;
  }
}

__global__ void inc_step_kernel(int* step) { *step += 1; }

int gap_adam_flat_devstep(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                          float eps, float weight_decay, int decoupled, int* step_dev, float grad_scale, void* stream) {
  GAP_CHECK_ARG(p && g && m && v && n > 0 && step_dev, "gap_adam_flat_devstep: bad arguments");
  if ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) |
       reinterpret_cast<uintptr_t>(v)) & 15) {
    set_error("gap_adam_flat_devstep: buffers must be 16-byte aligned");
    return GAP_ERR_ALIGNMENT;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  inc_step_kernel<<<1, 1, 0, st>>>(step_dev);
  adam_kernel<<<grid_for(n / 4 + 1, 256), 256, 0, st>>>(p, g, m, v, n, lr, beta1, beta2, eps, weight_decay, decoupled,
                                                        1.f, 1.f, grad_scale, step_dev);
  GAP_LAUNCH_CHECK();
  return 0;
}

int gap_gan_losses(double* acc4, double count, double l1_weight, double numel, double* out2, void* stream) {
  GAP_CHECK_ARG(acc4 && out2 && count > 0 && numel > 0, "gap_gan_losses: bad arguments");
  gan_losses_kernel<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(acc4, 1.0 / count, l1_weight / numel, out2);
  GAP_LAUNCH_CHECK();
  return 0;
}

int gap_pack_weights(const float* w, void* out, int mode, int n_phase, int rows, int rows_pad, int taps_h,
                     int taps_w, int c, int c_pad, int krow, int64_t s_r, int64_t s_c, int64_t s_kh, int64_t s_kw,
                     int kdim, void* stream) {
  GAP_CHECK_ARG(w && out && mode >= 0 && mode <= 3 && n_phase >= 1 && rows >= 1 && rows_pad >= rows && krow >= 1,
                "gap_pack_weights: bad arguments");
  GAP_CHECK_ARG(mode == 3 || (c_pad >= c && krow >= taps_h * taps_w * c_pad), "gap_pack_weights: krow too small");
  PackArgs a{w, static_cast<__nv_bfloat16*>(out), mode, n_phase, rows, rows_pad, taps_h, taps_w, c, c_pad, krow,
             s_r, s_c, s_kh, s_kw, kdim};
  const long long total = static_cast<long long>(n_phase) * rows_pad * krow;
  pack_weights_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
  GAP_LAUNCH_CHECK();
  return 0;
}

int gap_pack_weights_multi(const gap_pack_entry* table_dev, int n_entries, int total_tiles, void* stream) {
  GAP_CHECK_ARG(table_dev != nullptr && n_entries > 0 && total_tiles > 0, "gap_pack_weights_multi: empty table");
  pack_weights_multi_kernel<<<total_tiles, dim3(32, 8), 0, static_cast<cudaStream_t>(stream)>>>(table_dev, n_entries);
  GAP_LAUNCH_CHECK();
  return 0;
}

}  // extern "C"
