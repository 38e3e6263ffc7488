// Kernels the Siamese U-Net (models.py:47-145, train.py:34-128) needs beyond the shared conv / BatchNorm /
// Adam kernels: the 3-channel 3x3 im2col of its first conv, MaxPool2d(2), bilinear x2 upsampling with
// align_corners=True, the attention gate's elementwise pieces, 1x1 convolutions to a single channel
// (psi, conv_last) and the Dice / Focal / BCE loss family.  All of them are HBM-bound elementwise or
// reduction kernels: 16-byte vector accesses along the channel axis, warp-shuffle reductions, fp32 math.
#include <algorithm>

#include "common.h"
#include "ptx.cuh"

namespace gap {

typedef __nv_bfloat16 bf16;

__device__ __forceinline__ void unpack8(const uint4& raw, float (&v)[8]) {
  const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    v[2 * j] = bf16_lo(w[j]);
    v[2 * j + 1] = bf16_hi(w[j]);
  }
}
__device__ __forceinline__ uint4 pack8(const float (&v)[8]) {
  return make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
}

__device__ __forceinline__ void block_sum_to(double* dst, float v) {
  // sum v over the block and atomically add the total to *dst (fp64)
  __shared__ float red[32];
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  if (wid == 0) {
    float t = lane < ((blockDim.x + 31) >> 5) ? red[lane] : 0.f;
    t = warp_sum(t);
    if (lane == 0) atomicAdd(dst, static_cast<double>(t));
  }
}

// ------------------------------------------------------------------------------------------------
// im2col of Conv2d(C -> cout, k3, s1, p1), C = 1..4 (double_conv's first conv, models.py:9 via :54):
//   col[pix][(kh*3+kw)*C + c] = x[n, y-1+kh, x-1+kw, c]   (9*C values, zero padded to 64)
// x: NHWC bf16 with 4 channel slots per pixel.
// ------------------------------------------------------------------------------------------------
template <int C>
__global__ void im2col_k3s1p1_kernel(const bf16* __restrict__ x, long long ld, bf16* __restrict__ col, int n, int h,
                                     int w) {
  const long long total = static_cast<long long>(n) * h * w;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int px = static_cast<int>(i % w);
    const int py = static_cast<int>((i / w) % h);
    const long long img = i / (static_cast<long long>(w) * h);
    __align__(16) bf16 row[64];
#pragma unroll
    for (int k = 0; k < 64; ++k) row[k] = __float2bfloat16(0.f);
#pragma unroll
    for (int kh = 0; kh < 3; ++kh) {
      const int yy = py - 1 + kh;
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const int xx = px - 1 + kw;
        if (yy >= 0 && yy < h && xx >= 0 && xx < w) {
          const uint2 v = __ldg(reinterpret_cast<const uint2*>(x + ((img * h + yy) * w + xx) * ld));
          const bf16* pv = reinterpret_cast<const bf16*>(&v);
#pragma unroll
          for (int c = 0; c < C; ++c) row[(kh * 3 + kw) * C + c] = pv[c];
        }
      }
    }
    uint4* dst = reinterpret_cast<uint4*>(col + i * 64);
    const uint4* src = reinterpret_cast<const uint4*>(row);
#pragma unroll
    for (int k = 0; k < 8; ++k) dst[k] = src[k];
  }
}

// ------------------------------------------------------------------------------------------------
// MaxPool2d(2) (models.py:58) forward / backward, 8 channels per thread.  Backward routes the gradient to
// the first maximum in (kh, kw) scan order (torch's tie rule) and either writes or accumulates.
// ------------------------------------------------------------------------------------------------
__global__ void maxpool2x2_fwd_kernel(const bf16* __restrict__ x, long long ldx, bf16* __restrict__ out, long long ldo,
                                      int n, int h, int w, int c) {
  const int cv = c >> 3, ho = h >> 1, wo = w >> 1;
  const long long total = static_cast<long long>(n) * ho * wo * cv;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c8 = static_cast<int>(i % cv) << 3;
    long long r = i / cv;
    const int ox = static_cast<int>(r % wo);
    r /= wo;
    const int oy = static_cast<int>(r % ho);
    const long long img = r / ho;
    float m[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) m[j] = -INFINITY;
#pragma unroll
    for (int kh = 0; kh < 2; ++kh)
#pragma unroll
      for (int kw = 0; kw < 2; ++kw) {
        float v[8];
        unpack8(__ldg(reinterpret_cast<const uint4*>(x + ((img * h + 2 * oy + kh) * w + 2 * ox + kw) * ldx + c8)), v);
#pragma unroll
        for (int j = 0; j < 8; ++j) m[j] = v[j] > m[j] ? v[j] : m[j];
      }
    *reinterpret_cast<uint4*>(out + ((img * ho + oy) * wo + ox) * ldo + c8) = pack8(m);
  }
}

__global__ void maxpool2x2_bwd_kernel(const bf16* __restrict__ x, long long ldx, const bf16* __restrict__ gout,
                                      long long ldg, bf16* __restrict__ gin, long long ldi, int n, int h, int w, int c,
                                      int accumulate) {
  const int cv = c >> 3, ho = h >> 1, wo = w >> 1;
  const long long total = static_cast<long long>(n) * ho * wo * cv;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c8 = static_cast<int>(i % cv) << 3;
    long long r = i / cv;
    const int ox = static_cast<int>(r % wo);
    r /= wo;
    const int oy = static_cast<int>(r % ho);
    const long long img = r / ho;
    float v[4][8], g[8];
#pragma unroll
    for (int k = 0; k < 4; ++k)
      unpack8(__ldg(reinterpret_cast<const uint4*>(x + ((img * h + 2 * oy + (k >> 1)) * w + 2 * ox + (k & 1)) * ldx + c8)), v[k]);
    unpack8(__ldg(reinterpret_cast<const uint4*>(gout + ((img * ho + oy) * wo + ox) * ldg + c8)), g);
    int arg[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float m = v[0][j];
      arg[j] = 0;
#pragma unroll
      for (int k = 1; k < 4; ++k)
        if (v[k][j] > m) {
          m = v[k][j];
          arg[j] = k;
        }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      bf16* dst = gin + ((img * h + 2 * oy + (k >> 1)) * w + 2 * ox + (k & 1)) * ldi + c8;
      float o[8];
      if (accumulate) unpack8(*reinterpret_cast<const uint4*>(dst), o);
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = (accumulate ? o[j] : 0.f) + (arg[j] == k ? g[j] : 0.f);
      *reinterpret_cast<uint4*>(dst) = pack8(o);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// nn.Upsample(scale_factor=2, mode='bilinear', align_corners=True) (models.py:64): src = dst*(in-1)/(out-1)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void src_index(int o, int in_size, float scale, int& i0, int& i1, float& l) {
  const float s = scale * o;
  i0 = static_cast<int>(s);
  if (i0 > in_size - 1) i0 = in_size - 1;
  i1 = i0 + (i0 < in_size - 1 ? 1 : 0);
  l = s - i0;
}

// Work decomposition shared by both directions: a unit is a 1024-element segment of one image row (element = 8
// channels of one pixel), blocks stride over units.  Everything that depends on the row only (image, source rows and
// their weights) is computed once per unit, and the per-element index math is 32-bit (the flat 64-bit index with three
// divisions per element made these kernels instruction-bound: 2.6x / 4.3x their HBM time).
constexpr int kUpSeg = 1024;

__global__ void __launch_bounds__(256) upsample2x_fwd_kernel(const bf16* __restrict__ x, long long ldx,
                                                             bf16* __restrict__ out, long long ldo, int n, int h, int w,
                                                             int c, int cv_shift) {
  const int cv = c >> 3, ho = 2 * h, wo = 2 * w;
  const float sh = ho > 1 ? static_cast<float>(h - 1) / (ho - 1) : 0.f;
  const float sw = wo > 1 ? static_cast<float>(w - 1) / (wo - 1) : 0.f;
  const int per_row = wo * cv;
  const int segs = (per_row + kUpSeg - 1) / kUpSeg;
  const int units = n * ho * segs;
  for (int unit = blockIdx.x; unit < units; unit += gridDim.x) {
    const int row = unit / segs, seg = unit - row * segs;
    const int img = row / ho, oy = row - img * ho;
    int y0, y1;
    float ly;
    src_index(oy, h, sh, y0, y1, ly);
    const bf16* r0 = x + (static_cast<long long>(img) * h + y0) * w * ldx;
    const bf16* r1 = x + (static_cast<long long>(img) * h + y1) * w * ldx;
    bf16* ro = out + static_cast<long long>(row) * wo * ldo;
    const int j_end = min(per_row, (seg + 1) * kUpSeg);
    for (int j = seg * kUpSeg + threadIdx.x; j < j_end; j += blockDim.x) {
      const int ox = cv_shift >= 0 ? (j >> cv_shift) : (j / cv);
      const int c8 = (j - ox * cv) << 3;
      int x0, x1;
      float lx;
      src_index(ox, w, sw, x0, x1, lx);
      float a[8], b[8], cc[8], d[8], o[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(r0 + x0 * ldx + c8)), a);
      unpack8(__ldg(reinterpret_cast<const uint4*>(r0 + x1 * ldx + c8)), b);
      unpack8(__ldg(reinterpret_cast<const uint4*>(r1 + x0 * ldx + c8)), cc);
      unpack8(__ldg(reinterpret_cast<const uint4*>(r1 + x1 * ldx + c8)), d);
      const float w00 = (1.f - ly) * (1.f - lx), w01 = (1.f - ly) * lx, w10 = ly * (1.f - lx), w11 = ly * lx;
#pragma unroll
      for (int k = 0; k < 8; ++k) o[k] = w00 * a[k] + w01 * b[k] + w10 * cc[k] + w11 * d[k];
      *reinterpret_cast<uint4*>(ro + ox * ldo + c8) = pack8(o);
    }
  }
}

// weight with which output index o reads input index i (0 when it does not)
__device__ __forceinline__ float up_weight(int o, int i, int in_size, float scale) {
  int i0, i1;
  float l;
  src_index(o, in_size, scale, i0, i1, l);
  return (i0 == i ? 1.f - l : 0.f) + (i1 == i ? l : 0.f);
}
// [a, b]: the output indices that read input index i (src in (i-1, i+1): at most five of them at scale ~1/2;
// the scan covers two more on either side against rounding of the division)
__device__ __forceinline__ void up_contrib_range(int i, int in_size, int out_size, float scale, int& a, int& b) {
  if (scale == 0.f) {   // a single input row / column feeds every output
    a = 0;
    b = out_size - 1;
    return;
  }
  const int lo = max(0, static_cast<int>((i - 1) / scale) - 1);
  a = out_size;
  b = -1;
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    const int o = lo + k;
    if (o < out_size && up_weight(o, i, in_size, scale) != 0.f) {
      a = min(a, o);
      b = max(b, o);
    }
  }
}

// backward as a gather: input pixel (iy, ix) collects from the (few) output pixels whose footprint holds it
__global__ void __launch_bounds__(256) upsample2x_bwd_kernel(const bf16* __restrict__ gout, long long ldg,
                                                             bf16* __restrict__ gin, long long ldi, int n, int h, int w,
                                                             int c, int accumulate, int cv_shift) {
  const int cv = c >> 3, ho = 2 * h, wo = 2 * w;
  const float sh = ho > 1 ? static_cast<float>(h - 1) / (ho - 1) : 0.f;
  const float sw = wo > 1 ? static_cast<float>(w - 1) / (wo - 1) : 0.f;
  const int per_row = w * cv;
  const int segs = (per_row + kUpSeg - 1) / kUpSeg;
  const int units = n * h * segs;
  for (int unit = blockIdx.x; unit < units; unit += gridDim.x) {
    const int row = unit / segs, seg = unit - row * segs;
    const int img = row / h, iy = row - img * h;
    int ya, yb;
    up_contrib_range(iy, h, ho, sh, ya, yb);
    bf16* ri = gin + static_cast<long long>(row) * w * ldi;
    const int j_end = min(per_row, (seg + 1) * kUpSeg);
    for (int j = seg * kUpSeg + threadIdx.x; j < j_end; j += blockDim.x) {
      const int ix = cv_shift >= 0 ? (j >> cv_shift) : (j / cv);
      const int c8 = (j - ix * cv) << 3;
      int xa, xb;
      up_contrib_range(ix, w, wo, sw, xa, xb);
      float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      for (int oy = ya; oy <= yb; ++oy) {
        const float wy = up_weight(oy, iy, h, sh);
        const bf16* rg = gout + (static_cast<long long>(img) * ho + oy) * wo * ldg + c8;
        for (int ox = xa; ox <= xb; ++ox) {
          const float wgt = wy * up_weight(ox, ix, w, sw);
          float g[8];
          unpack8(__ldg(reinterpret_cast<const uint4*>(rg + ox * ldg)), g);
#pragma unroll
          for (int k = 0; k < 8; ++k) acc[k] += wgt * g[k];
        }
      }
      bf16* dst = ri + ix * ldi + c8;
      if (accumulate) {
        float o[8];
        unpack8(*reinterpret_cast<const uint4*>(dst), o);
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[k] += o[k];
      }
      *reinterpret_cast<uint4*>(dst) = pack8(acc);
    }
  }
}

// nn.Dropout(p) (models.py:198) in place on a bf16 [pixels][c] tensor (channel slice allowed): x = keep ? x/(1-p) : 0,
// keep decided by a counter-based hash of (seed, offset + element index), so forward and backward regenerate the
// same mask without storing it (the backward applies the same kernel to the gradient).
__device__ __forceinline__ uint32_t mix32(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return static_cast<uint32_t>((z ^ (z >> 31)) >> 32);
}
__global__ void dropout_kernel(bf16* __restrict__ x, long long ld, long long pixels, int c, float p_drop, float scale,
                               unsigned long long seed, unsigned long long offset) {
  const int cv = c >> 3;
  const long long total = pixels * cv;
  const uint32_t thresh = static_cast<uint32_t>(fminf(p_drop, 0.999999f) * 4294967296.0f);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long pix = i / cv;
    const int c8 = static_cast<int>(i - pix * cv) << 3;
    float v[8];
    unpack8(*reinterpret_cast<const uint4*>(x + pix * ld + c8), v);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint64_t idx = static_cast<uint64_t>(pix) * c + c8 + j;
      const bool keep = mix32(seed * 0xD1342543DE82EF95ull + offset + idx) >= thresh;
      v[j] = keep ? v[j] * scale : 0.f;
    }
    *reinterpret_cast<uint4*>(x + pix * ld + c8) = pack8(v);
  }
}

// ------------------------------------------------------------------------------------------------
// AttentionGate (models.py:18-44) elementwise pieces
//   s   = ReLU(BN_g(yg) + BN_x(yx))                        (add_relu)
//   psi = Sigmoid(BN_psi(ypsi)),  out = x * psi            (gate)
// ------------------------------------------------------------------------------------------------
__global__ void att_add_relu_fwd_kernel(const bf16* __restrict__ yg, const float* __restrict__ scg,
                                        const float* __restrict__ shg, const bf16* __restrict__ yx,
                                        const float* __restrict__ scx, const float* __restrict__ shx,
                                        bf16* __restrict__ s, long long pixels, int c) {
  const int cv = c >> 3;
  const long long total = pixels * cv;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c8 = static_cast<int>(i % cv) << 3;
    float a[8], b[8], o[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(yg + i * 8)), a);
    unpack8(__ldg(reinterpret_cast<const uint4*>(yx + i * 8)), b);
#pragma unroll
    for (int j = 0; j < 8; ++j)
      o[j] = fmaxf(fmaf(a[j], scg[c8 + j], shg[c8 + j]) + fmaf(b[j], scx[c8 + j], shx[c8 + j]), 0.f);
    *reinterpret_cast<uint4*>(s + i * 8) = pack8(o);
  }
}

// d = (s > 0) ? gs : 0   (gradient at both BatchNorm outputs)
__global__ void relu_bwd_kernel(const bf16* __restrict__ s, const bf16* __restrict__ gs, bf16* __restrict__ d,
                                long long n8) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    float a[8], g[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(s + i * 8)), a);
    unpack8(__ldg(reinterpret_cast<const uint4*>(gs + i * 8)), g);
#pragma unroll
    for (int j = 0; j < 8; ++j) g[j] = a[j] > 0.f ? g[j] : 0.f;
    *reinterpret_cast<uint4*>(d + i * 8) = pack8(g);
  }
}

// LeakyReLU backward with strided operands: d (+)= y > 0 ? g : slope * g   (y = the activation's output or input: same sign)
__global__ void lrelu_bwd_kernel(const bf16* __restrict__ y, long long ldy, const bf16* __restrict__ g, long long ldg,
                                 float slope, bf16* __restrict__ d, long long ldd, long long pixels, int c, int accumulate) {
  const int cv = c >> 3;
  const long long total = pixels * cv;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long pix = i / cv;
    const int c8 = static_cast<int>(i - pix * cv) << 3;
    float a[8], b[8], o[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(y + pix * ldy + c8)), a);
    unpack8(__ldg(reinterpret_cast<const uint4*>(g + pix * ldg + c8)), b);
    if (accumulate) unpack8(*reinterpret_cast<const uint4*>(d + pix * ldd + c8), o);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float v = a[j] > 0.f ? b[j] : slope * b[j];
      o[j] = accumulate ? o[j] + v : v;
    }
    *reinterpret_cast<uint4*>(d + pix * ldd + c8) = pack8(o);
  }
}

// psi = sigmoid(ypsi*scale + shift); out[pix][c] = x[pix][c] * psi[pix]
__global__ void att_gate_fwd_kernel(const float* __restrict__ ypsi, const float* __restrict__ scale,
                                    const float* __restrict__ shift, float* __restrict__ psi, const bf16* __restrict__ x,
                                    long long ldx, bf16* __restrict__ out, long long ldo, long long pixels, int c) {
  const int cv = c >> 3;
  const long long total = pixels * cv;
  const float sc = scale[0], sh = shift[0];
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long pix = i / cv;
    const int c8 = static_cast<int>(i - pix * cv) << 3;
    const float p = 1.f / (1.f + __expf(-fmaf(ypsi[pix], sc, sh)));
    if (c8 == 0) psi[pix] = p;
    float v[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(x + pix * ldx + c8)), v);
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] *= p;
    *reinterpret_cast<uint4*>(out + pix * ldo + c8) = pack8(v);
  }
}

// gate backward: gx (+)= gout * psi;  dz[pix] = (sum_c gout*x) * psi*(1-psi)   (gradient at BN_psi's output)
// 8 lanes per pixel (16 bytes each per step), shuffle-reduced.
__global__ void att_gate_bwd_kernel(const bf16* __restrict__ gout, long long ldg, const bf16* __restrict__ x,
                                    long long ldx, const float* __restrict__ psi, bf16* __restrict__ gx, long long ldgx,
                                    int accumulate, float* __restrict__ dz, long long pixels, int c) {
  const int sub = threadIdx.x & 7;
  const long long pix0 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 3;
  const long long stride = ((long long)gridDim.x * blockDim.x) >> 3;
  for (long long pix = pix0; pix < pixels; pix += stride) {   // all 8 lanes of a pixel share `pix`
    const float p = psi[pix];
    float dot = 0.f;
    for (int c8 = sub * 8; c8 < c; c8 += 64) {
      float g[8], v[8], o[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(gout + pix * ldg + c8)), g);
      unpack8(__ldg(reinterpret_cast<const uint4*>(x + pix * ldx + c8)), v);
      if (accumulate) unpack8(*reinterpret_cast<const uint4*>(gx + pix * ldgx + c8), o);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        dot += g[j] * v[j];
        o[j] = (accumulate ? o[j] : 0.f) + g[j] * p;
      }
      *reinterpret_cast<uint4*>(gx + pix * ldgx + c8) = pack8(o);
    }
    dot += __shfl_xor_sync(0xffffffffu, dot, 1);
    dot += __shfl_xor_sync(0xffffffffu, dot, 2);
    dot += __shfl_xor_sync(0xffffffffu, dot, 4);
    if (sub == 0) dz[pix] = dot * p * (1.f - p);
  }
}

// ------------------------------------------------------------------------------------------------
// Single-channel fp32 maps (psi path, conv_last logits): BatchNorm statistics and backward
// ------------------------------------------------------------------------------------------------
__global__ void vec_stats_kernel(const float* __restrict__ y, long long n, double* __restrict__ stats) {
  float s = 0.f, q = 0.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float v = y[i];
    s += v;
    q += v * v;
  }
  block_sum_to(stats, s);
  block_sum_to(stats + 1, q);
}
// sums[0] += sum dz, sums[1] += sum dz * xhat
__global__ void vec_bn_bwd_reduce_kernel(const float* __restrict__ y, const float* __restrict__ dz, long long n,
                                         const float* __restrict__ mean, const float* __restrict__ invstd,
                                         double* __restrict__ sums) {
  const float mu = mean[0], is = invstd[0];
  float s = 0.f, q = 0.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float d = dz[i];
    s += d;
    q += d * (y[i] - mu) * is;
  }
  block_sum_to(sums, s);
  block_sum_to(sums + 1, q);
}
// dy = scale * (dz - m1 - xhat * m2)
__global__ void vec_bn_bwd_apply_kernel(const float* __restrict__ y, const float* __restrict__ dz, long long n,
                                        const float* __restrict__ scale, const float* __restrict__ mean,
                                        const float* __restrict__ invstd, const double* __restrict__ sums,
                                        double inv_count, float* __restrict__ dy) {
  const float sc = scale[0], mu = mean[0], is = invstd[0];
  const float m1 = static_cast<float>(sums[0] * inv_count), m2 = static_cast<float>(sums[1] * inv_count);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    dy[i] = sc * (dz[i] - m1 - (y[i] - mu) * is * m2);
}

// ------------------------------------------------------------------------------------------------
// Conv2d(C -> 1, k1) + bias (psi's conv models.py:32, conv_last models.py:90): fp32 output map
// ------------------------------------------------------------------------------------------------
__global__ void conv1x1_cout1_fwd_kernel(const bf16* __restrict__ x, long long ldx, const float* __restrict__ w,
                                         const float* __restrict__ bias, float* __restrict__ out, long long pixels, int c) {
  const int sub = threadIdx.x & 7;
  const long long pix0 = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 3;
  const long long stride = ((long long)gridDim.x * blockDim.x) >> 3;
  const float b = bias ? bias[0] : 0.f;
  for (long long pix = pix0; pix < pixels; pix += stride) {
    float dot = 0.f;
    for (int c8 = sub * 8; c8 < c; c8 += 64) {
      float v[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(x + pix * ldx + c8)), v);
#pragma unroll
      for (int j = 0; j < 8; ++j) dot += v[j] * __bfloat162float(__float2bfloat16(__ldg(w + c8 + j)));
    }
    dot += __shfl_xor_sync(0xffffffffu, dot, 1);
    dot += __shfl_xor_sync(0xffffffffu, dot, 2);
    dot += __shfl_xor_sync(0xffffffffu, dot, 4);
    if (sub == 0) out[pix] = dot + b;
  }
}
// gx[pix][c] = dl[pix] * w[c]
__global__ void conv1x1_cout1_dgrad_kernel(const float* __restrict__ dl, const float* __restrict__ w,
                                           bf16* __restrict__ gx, long long ldg, long long pixels, int c) {
  const int cv = c >> 3;
  const long long total = pixels * cv;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long pix = i / cv;
    const int c8 = static_cast<int>(i - pix * cv) << 3;
    const float d = dl[pix];
    float o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = d * __bfloat162float(__float2bfloat16(__ldg(w + c8 + j)));
    *reinterpret_cast<uint4*>(gx + pix * ldg + c8) = pack8(o);
  }
}
// dw[c] += sum_pix dl[pix] * x[pix][c];  db += sum dl      (blockDim = (c/8 lanes, pixel lanes))
__global__ void conv1x1_cout1_wgrad_kernel(const float* __restrict__ dl, const bf16* __restrict__ x, long long ldx,
                                           long long pixels, int c, float* __restrict__ dw, float* __restrict__ db) {
  extern __shared__ float sm[];  // [blockDim.y][c]
  const int cv = c >> 3;
  float bsum = 0.f;
  for (int cg = threadIdx.x; cg < cv; cg += blockDim.x) {
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (long long pix = blockIdx.x * (long long)blockDim.y + threadIdx.y; pix < pixels;
         pix += (long long)gridDim.x * blockDim.y) {
      const float d = dl[pix];
      float v[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(x + pix * ldx + cg * 8)), v);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += d * v[j];
      if (cg == 0) bsum += d;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) sm[threadIdx.y * c + cg * 8 + j] = acc[j];
  }
  __syncthreads();
  const int tid = threadIdx.y * blockDim.x + threadIdx.x, nthr = blockDim.x * blockDim.y;
  for (int ch = tid; ch < c; ch += nthr) {
    float t = 0.f;
    for (int r = 0; r < blockDim.y; ++r) t += sm[r * c + ch];
    atomicAdd(dw + ch, t);
  }
  if (db != nullptr && threadIdx.x == 0) {
    // threads with threadIdx.x == 0 own channel group 0 and therefore the bias partials
    atomicAdd(db, bsum);
  }
}

// ------------------------------------------------------------------------------------------------
// Segmentation losses (train.py:34-128) on fp32 logits [n] against int64 labels {0,1}:
//   p = sigmoid(x), t = float(label)
//   Dice  = 1 - (2*sum(p t) + s) / (sum p + sum t + s)                                  (train.py:40-45)
//   BCEw  = mean(pw*t*softplus(-x) + (1-t)*softplus(x))                                 (train.py:86,94)
//   Focal = mean(a_t * (1 - exp(-bce))^gamma * bce), bce unweighted, a_t = t*a + (1-t)(1-a)   (train.py:67-73)
// mode 0: CombinedLoss = alpha*BCEw + (1-alpha)*Dice (train.py:82-105);  mode 1: FocalDiceLoss = beta*Focal + (1-beta)*Dice
// pass 1 accumulates sums[0..3] = sum p*t, sum p, sum t, sum of the pointwise term; pass 2 writes the loss and the gradient.
// ------------------------------------------------------------------------------------------------
struct SegLossArgs {
  const float* x;
  const long long* labels;
  long long n;
  int mode;
  float w_point, w_dice;   // alpha / (1-alpha)  or  beta / (1-beta)
  float pos_weight, smooth, gamma, focal_alpha;
  double* sums;            // [4], zeroed by the caller (pass 2 re-zeroes)
  float* grad;             // d(loss)/d(logit), may be NULL
  double* loss;            // [1] written (not accumulated)
  float grad_scale;
};

__device__ __forceinline__ float softplus_f(float v) { return fmaxf(v, 0.f) + log1pf(__expf(-fabsf(v))); }

__global__ void seg_loss_reduce_kernel(const SegLossArgs a) {
  float spt = 0.f, sp = 0.f, st = 0.f, sl = 0.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < a.n; i += (long long)gridDim.x * blockDim.x) {
    const float x = a.x[i];
    const float t = a.labels[i] != 0 ? 1.f : 0.f;
    const float p = 1.f / (1.f + __expf(-x));
    spt += p * t;
    sp += p;
    st += t;
    if (a.mode == 0) {
      sl += a.pos_weight * t * softplus_f(-x) + (1.f - t) * softplus_f(x);
    } else {
      const float bce = t * softplus_f(-x) + (1.f - t) * softplus_f(x);
      const float pt = __expf(-bce);
      const float at = t * a.focal_alpha + (1.f - t) * (1.f - a.focal_alpha);
      sl += at * __powf(fmaxf(1.f - pt, 0.f), a.gamma) * bce;
    }
  }
  block_sum_to(a.sums + 0, spt);
  block_sum_to(a.sums + 1, sp);
  block_sum_to(a.sums + 2, st);
  block_sum_to(a.sums + 3, sl);
}

__global__ void seg_loss_grad_kernel(const SegLossArgs a) {
  const double I = a.sums[0], P = a.sums[1], T = a.sums[2], L = a.sums[3];
  const double D = P + T + a.smooth;
  const double dice = 1.0 - (2.0 * I + a.smooth) / D;
  if (blockIdx.x == 0 && threadIdx.x == 0) a.loss[0] = a.w_point * (L / static_cast<double>(a.n)) + a.w_dice * dice;
  if (a.grad != nullptr) {
    const float inv_n = 1.f / static_cast<float>(a.n);
    const float num = static_cast<float>(2.0 * I + a.smooth), fD = static_cast<float>(D);
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < a.n; i += (long long)gridDim.x * blockDim.x) {
      const float x = a.x[i];
      const float t = a.labels[i] != 0 ? 1.f : 0.f;
      const float p = 1.f / (1.f + __expf(-x));
      // d(dice)/dp_i = -(2 t D - (2I+s)) / D^2
      const float ddice = -(2.f * t * fD - num) / (fD * fD) * p * (1.f - p);
      float dpoint;
      if (a.mode == 0) {
        dpoint = (-a.pos_weight * t * (1.f - p) + (1.f - t) * p) * inv_n;
      } else {
        const float bce = t * softplus_f(-x) + (1.f - t) * softplus_f(x);
        const float pt = __expf(-bce);
        const float om = fmaxf(1.f - pt, 0.f);
        const float at = t * a.focal_alpha + (1.f - t) * (1.f - a.focal_alpha);
        const float dbce = p - t;
        const float f1 = om > 0.f ? a.gamma * __powf(om, a.gamma - 1.f) * pt * bce : 0.f;
        dpoint = at * dbce * (f1 + __powf(om, a.gamma)) * inv_n;
      }
      a.grad[i] = a.grad_scale * (a.w_point * dpoint + a.w_dice * ddice);
    }
  }
}
__global__ void zero4_kernel(double* s) {
  if (threadIdx.x < 4) s[threadIdx.x] = 0.0;
}

static inline int grid_of(long long work, int block, int max_blocks) {
  long long g = (work + block - 1) / block;
  if (g < 1) g = 1;
  return static_cast<int>(g < max_blocks ? g : max_blocks);
}
// log2(v) when v is a power of two, else -1 (the kernels then divide)
static inline int pow2_shift(int v) {
  int s = 0;
  while ((1 << s) < v) ++s;
  return (1 << s) == v ? s : -1;
}
static inline long long up_segments(int row_pixels, int c) {
  return (static_cast<long long>(row_pixels) * (c / 8) + kUpSeg - 1) / kUpSeg;
}

}  // namespace gap

using namespace gap;

#define SI_LAUNCH_OK()            \
  do {                            \
    GAP_CUDA(cudaGetLastError()); \
    return 0;                     \
  } while (0)

// evaluate.py:34-64 (calculate_metrics) on the device: preds = sigmoid(logits) > 0.5 against {0,1} labels, one
// [TP, FP, FN, TN] count row per sample (the reference loops over samples and moves every map to the CPU first).
// gridDim.y = samples; counts are accumulated (+=) so a caller can sum over batches.
__global__ void seg_confusion_kernel(const float* __restrict__ logits, const long long* __restrict__ lab_i64,
                                     const float* __restrict__ lab_f32, long long hw,
                                     unsigned long long* __restrict__ counts) {
  const long long base = static_cast<long long>(blockIdx.y) * hw;
  unsigned int c[4] = {0u, 0u, 0u, 0u};
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < hw;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float x = logits[base + i];
    // the reference thresholds the fp32 sigmoid, not the logit: logits in (0, ~6e-8] round to exactly 0.5 -> negative
    const bool pred = 1.f / (1.f + expf(-x)) > 0.5f;
    const bool tgt = lab_i64 ? lab_i64[base + i] != 0 : lab_f32[base + i] != 0.f;
    if (pred && tgt) ++c[0];
    else if (pred && !tgt) ++c[1];
    else if (!pred && tgt) ++c[2];
    else ++c[3];
  }
  __shared__ unsigned int red[4][8];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    unsigned int v = c[k];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[k][wid] = v;
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    unsigned long long tot = 0;
    for (int w2 = 0; w2 < static_cast<int>(blockDim.x >> 5); ++w2) tot += red[threadIdx.x][w2];
    if (tot) atomicAdd(counts + blockIdx.y * 4 + threadIdx.x, tot);
  }
}

extern "C" {

int gap_im2col_k3s1p1_c3(const void* x, int64_t ld, void* col, int n, int h, int w, void* stream) {
  GAP_CHECK_ARG(x && col && n > 0 && h > 0 && w > 0 && ld % 4 == 0, "gap_im2col_k3s1p1_c3: bad arguments");
  return gap_im2col_k3s1p1_c(x, ld, 3, col, n, h, w, stream);
}

int gap_im2col_k3s1p1_c(const void* x, int64_t ld, int c, void* col, int n, int h, int w, void* stream) {
  GAP_CHECK_ARG(c >= 1 && c <= 4, "gap_im2col_k3s1p1_c: c must be 1..4");
  GAP_CHECK_ARG(x && col && n > 0 && h > 0 && w > 0 && ld % 4 == 0, "gap_im2col_k3s1p1_c: bad arguments");
  const long long total = static_cast<long long>(n) * h * w;
  const int grid = grid_of(total, 128, 148 * 16);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bf16* xi = static_cast<const bf16*>(x);
  bf16* co = static_cast<bf16*>(col);
  switch (c) {
    case 1: im2col_k3s1p1_kernel<1><<<grid, 128, 0, st>>>(xi, ld, co, n, h, w); break;
    case 2: im2col_k3s1p1_kernel<2><<<grid, 128, 0, st>>>(xi, ld, co, n, h, w); break;
    case 3: im2col_k3s1p1_kernel<3><<<grid, 128, 0, st>>>(xi, ld, co, n, h, w); break;
    default: im2col_k3s1p1_kernel<4><<<grid, 128, 0, st>>>(xi, ld, co, n, h, w); break;
  }
  SI_LAUNCH_OK();
}

int gap_maxpool2x2_fwd(const void* x, int64_t ldx, void* out, int64_t ldo, int n, int h, int w, int c, void* stream) {
  GAP_CHECK_ARG(x && out && n > 0 && h > 1 && w > 1 && h % 2 == 0 && w % 2 == 0 && c % 8 == 0 && ldx % 8 == 0 && ldo % 8 == 0,
                "gap_maxpool2x2_fwd: bad arguments");
  const long long total = static_cast<long long>(n) * (h / 2) * (w / 2) * (c / 8);
  maxpool2x2_fwd_kernel<<<grid_of(total, 256, 148 * 16), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const bf16*>(x), ldx, static_cast<bf16*>(out), ldo, n, h, w, c);
  SI_LAUNCH_OK();
}

int gap_maxpool2x2_bwd(const void* x, int64_t ldx, const void* gout, int64_t ldg, void* gin, int64_t ldi, int n, int h,
                       int w, int c, int accumulate, void* stream) {
  GAP_CHECK_ARG(x && gout && gin && n > 0 && h % 2 == 0 && w % 2 == 0 && c % 8 == 0 && ldx % 8 == 0 && ldg % 8 == 0 && ldi % 8 == 0,
                "gap_maxpool2x2_bwd: bad arguments");
  const long long total = static_cast<long long>(n) * (h / 2) * (w / 2) * (c / 8);
  maxpool2x2_bwd_kernel<<<grid_of(total, 256, 148 * 16), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const bf16*>(x), ldx, static_cast<const bf16*>(gout), ldg, static_cast<bf16*>(gin), ldi, n, h, w, c,
      accumulate);
  SI_LAUNCH_OK();
}

int gap_upsample_bilinear2x_fwd(const void* x, int64_t ldx, void* out, int64_t ldo, int n, int h, int w, int c,
                                void* stream) {
  GAP_CHECK_ARG(x && out && n > 0 && h > 0 && w > 0 && c % 8 == 0 && ldx % 8 == 0 && ldo % 8 == 0,
                "gap_upsample_bilinear2x_fwd: bad arguments");
  const long long units = static_cast<long long>(n) * (2 * h) * up_segments(2 * w, c);
  GAP_CHECK_ARG(units < (1ll << 31) && static_cast<long long>(2 * w) * (c / 8) < (1ll << 30),
                "gap_upsample_bilinear2x_fwd: tensor too large");
  upsample2x_fwd_kernel<<<grid_of(units, 1, 148 * 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const bf16*>(x), ldx, static_cast<bf16*>(out), ldo, n, h, w, c, pow2_shift(c / 8));
  SI_LAUNCH_OK();
}

int gap_upsample_bilinear2x_bwd(const void* gout, int64_t ldg, void* gin, int64_t ldi, int n, int h, int w, int c,
                                int accumulate, void* stream) {
  GAP_CHECK_ARG(gout && gin && n > 0 && h > 0 && w > 0 && c % 8 == 0 && ldg % 8 == 0 && ldi % 8 == 0,
                "gap_upsample_bilinear2x_bwd: bad arguments");
  const long long units = static_cast<long long>(n) * h * up_segments(w, c);
  GAP_CHECK_ARG(units < (1ll << 31) && static_cast<long long>(w) * (c / 8) < (1ll << 30),
                "gap_upsample_bilinear2x_bwd: tensor too large");
  upsample2x_bwd_kernel<<<grid_of(units, 1, 148 * 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const bf16*>(gout), ldg, static_cast<bf16*>(gin), ldi, n, h, w, c, accumulate, pow2_shift(c / 8));
  SI_LAUNCH_OK();
}

int gap_dropout_bf16(void* x, int64_t ld, int64_t pixels, int c, float p_drop, uint64_t seed, uint64_t offset, void* stream) {
  GAP_CHECK_ARG(x && pixels > 0 && c % 8 == 0 && ld % 8 == 0 && p_drop >= 0.f && p_drop < 1.f, "gap_dropout_bf16: bad arguments");
  dropout_kernel<<<grid_of(pixels * (c / 8), 256, 148 * 16), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<bf16*>(x), ld, pixels, c, p_drop, 1.f / (1.f - p_drop), seed, offset);
  SI_LAUNCH_OK();
}

int gap_att_add_relu_fwd(const void* yg, const float* scale_g, const float* shift_g, const void* yx, const float* scale_x,
                         const float* shift_x, void* s, int64_t pixels, int c, void* stream) {
  GAP_CHECK_ARG(yg && yx && s && scale_g && shift_g && scale_x && shift_x && pixels > 0 && c % 8 == 0,
                "gap_att_add_relu_fwd: bad arguments");
  att_add_relu_fwd_kernel<<<grid_of(pixels * (c / 8), 256, 148 * 16), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const bf16*>(yg), scale_g, shift_g, static_cast<const bf16*>(yx), scale_x, shift_x,
      static_cast<bf16*>(s), pixels, c);
  SI_LAUNCH_OK();
}

int gap_relu_bwd(const void* s, const void* gs, void* d, int64_t count, void* stream) {
  GAP_CHECK_ARG(s && gs && d && count > 0 && count % 8 == 0, "gap_relu_bwd: bad arguments");
  relu_bwd_kernel<<<grid_of(count / 8, 256, 148 * 16), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const bf16*>(s), static_cast<const bf16*>(gs), static_cast<bf16*>(d), count / 8);
  SI_LAUNCH_OK();
}

int gap_lrelu_bwd_bf16(const void* y, int64_t ldy, const void* g, int64_t ldg, float slope, void* d, int64_t ldd,
                       int64_t pixels, int c, int accumulate, void* stream) {
  GAP_CHECK_ARG(y && g && d && pixels > 0 && c > 0 && c % 8 == 0 && ldy % 8 == 0 && ldg % 8 == 0 && ldd % 8 == 0,
                "gap_lrelu_bwd_bf16: bad arguments");
  lrelu_bwd_kernel<<<grid_of(pixels * (c / 8), 256, 148 * 16), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const bf16*>(y), ldy, static_cast<const bf16*>(g), ldg, slope, static_cast<bf16*>(d), ldd, pixels, c,
      accumulate);
  SI_LAUNCH_OK();
}

int gap_att_gate_fwd(const float* ypsi, const float* scale, const float* shift, float* psi, const void* x, int64_t ldx,
                     void* out, int64_t ldo, int64_t pixels, int c, void* stream) {
  GAP_CHECK_ARG(ypsi && scale && shift && psi && x && out && pixels > 0 && c % 8 == 0 && ldx % 8 == 0 && ldo % 8 == 0,
                "gap_att_gate_fwd: bad arguments");
  att_gate_fwd_kernel<<<grid_of(pixels * (c / 8), 256, 148 * 16), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      ypsi, scale, shift, psi, static_cast<const bf16*>(x), ldx, static_cast<bf16*>(out), ldo, pixels, c);
  SI_LAUNCH_OK();
}

int gap_att_gate_bwd(const void* gout, int64_t ldg, const void* x, int64_t ldx, const float* psi, void* gx, int64_t ldgx,
                     int accumulate, float* dz, int64_t pixels, int c, void* stream) {
  GAP_CHECK_ARG(gout && x && psi && gx && dz && pixels > 0 && c % 8 == 0 && ldg % 8 == 0 && ldx % 8 == 0 && ldgx % 8 == 0,
                "gap_att_gate_bwd: bad arguments");
  att_gate_bwd_kernel<<<grid_of(pixels * 8, 256, 148 * 16), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const bf16*>(gout), ldg, static_cast<const bf16*>(x), ldx, psi, static_cast<bf16*>(gx), ldgx,
      accumulate, dz, pixels, c);
  SI_LAUNCH_OK();
}

int gap_vec_stats(const float* y, int64_t n, double* stats, void* stream) {
  GAP_CHECK_ARG(y && stats && n > 0, "gap_vec_stats: bad arguments");
  vec_stats_kernel<<<grid_of(n, 256, 148 * 4), 256, 0, static_cast<cudaStream_t>(stream)>>>(y, n, stats);
  SI_LAUNCH_OK();
}

int gap_vec_bn_bwd(const float* y, const float* dz, int64_t n, const float* scale, const float* mean, const float* invstd,
                   double* sums, float* dy, void* stream) {
  GAP_CHECK_ARG(y && dz && scale && mean && invstd && sums && dy && n > 0, "gap_vec_bn_bwd: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  vec_bn_bwd_reduce_kernel<<<grid_of(n, 256, 148 * 4), 256, 0, st>>>(y, dz, n, mean, invstd, sums);
  GAP_CUDA(cudaGetLastError());
  vec_bn_bwd_apply_kernel<<<grid_of(n, 256, 148 * 8), 256, 0, st>>>(y, dz, n, scale, mean, invstd, sums, 1.0 / n, dy);
  SI_LAUNCH_OK();
}

int gap_conv1x1_cout1_fwd(const void* x, int64_t ldx, const float* w, const float* bias, float* out, int64_t pixels, int c,
                          void* stream) {
  GAP_CHECK_ARG(x && w && out && pixels > 0 && c % 8 == 0 && ldx % 8 == 0, "gap_conv1x1_cout1_fwd: bad arguments");
  conv1x1_cout1_fwd_kernel<<<grid_of(pixels * 8, 256, 148 * 16), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const bf16*>(x), ldx, w, bias, out, pixels, c);
  SI_LAUNCH_OK();
}

int gap_conv1x1_cout1_dgrad(const float* dl, const float* w, void* gx, int64_t ldg, int64_t pixels, int c, void* stream) {
  GAP_CHECK_ARG(dl && w && gx && pixels > 0 && c % 8 == 0 && ldg % 8 == 0, "gap_conv1x1_cout1_dgrad: bad arguments");
  conv1x1_cout1_dgrad_kernel<<<grid_of(pixels * (c / 8), 256, 148 * 16), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      dl, w, static_cast<bf16*>(gx), ldg, pixels, c);
  SI_LAUNCH_OK();
}

int gap_conv1x1_cout1_wgrad(const float* dl, const void* x, int64_t ldx, int64_t pixels, int c, float* dw, float* db,
                            void* stream) {
  GAP_CHECK_ARG(dl && x && dw && pixels > 0 && c % 8 == 0 && c <= 4096 && ldx % 8 == 0, "gap_conv1x1_cout1_wgrad: bad arguments");
  const int cv = c / 8;
  int bx = cv < 64 ? cv : 64;
  int by = 256 / bx;
  dim3 block(bx, by);
  const size_t smem = static_cast<size_t>(by) * c * sizeof(float);
  if (smem > 48 * 1024) {
    set_error("gap_conv1x1_cout1_wgrad: %d channels need %zu bytes of shared memory", c, smem);
    return GAP_ERR_UNSUPPORTED;
  }
  const long long slabs = (pixels + by - 1) / by;
  const int grid = static_cast<int>(slabs < 148 * 4 ? slabs : 148 * 4);
  conv1x1_cout1_wgrad_kernel<<<grid, block, smem, static_cast<cudaStream_t>(stream)>>>(
      dl, static_cast<const bf16*>(x), ldx, pixels, c, dw, db);
  SI_LAUNCH_OK();
}

int gap_seg_loss(const float* logits, const int64_t* labels, int64_t n, int mode, float w_point, float w_dice,
                 float pos_weight, float smooth, float gamma, float focal_alpha, double* sums4, float* grad,
                 float grad_scale, double* loss, void* stream) {
  GAP_CHECK_ARG(logits && labels && sums4 && loss && n > 0 && (mode == 0 || mode == 1), "gap_seg_loss: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  SegLossArgs a{logits, reinterpret_cast<const long long*>(labels), n, mode, w_point, w_dice, pos_weight, smooth, gamma,
                focal_alpha, sums4, grad, loss, grad_scale};
  zero4_kernel<<<1, 32, 0, st>>>(sums4);
  seg_loss_reduce_kernel<<<grid_of(n, 256, 148 * 4), 256, 0, st>>>(a);
  GAP_CUDA(cudaGetLastError());
  seg_loss_grad_kernel<<<grid_of(n, 256, 148 * 8), 256, 0, st>>>(a);
  SI_LAUNCH_OK();
}

int gap_seg_confusion(const float* logits, const void* labels, int labels_are_i64, int n, int64_t hw, int64_t* counts,
                      void* stream) {
  GAP_CHECK_ARG(logits && labels && counts && n > 0 && hw > 0, "gap_seg_confusion: bad arguments");
  const int bx = static_cast<int>(std::min<long long>((hw + 255) / 256, 148 * 4 / std::max(1, std::min(n, 16)) + 1));
  dim3 grid(bx, n);
  seg_confusion_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      logits, labels_are_i64 ? static_cast<const long long*>(labels) : nullptr,
      labels_are_i64 ? nullptr : static_cast<const float*>(labels), hw, reinterpret_cast<unsigned long long*>(counts));
  SI_LAUNCH_OK();
}

}  // extern "C"
