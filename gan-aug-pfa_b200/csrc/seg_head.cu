// Multi-class head of the Siamese U-Net: SiameseUNet(n_channels, n_classes) with n_classes = K = 1..16
// (models.py:90 `conv_last = nn.Conv2d(64, n_classes, 1)`), nn.CrossEntropyLoss on its output, the softmax CE / focal
// + multi-class Dice losses and the per-sample K x K confusion matrix.
//
// Layout: the logits and their gradient are fp32 class planes [n][K][hw] (NCHW, what nn.CrossEntropyLoss and
// torch.argmax(dim=1) expect); for K = 1 that is the [n][hw] map of the single-class path.  The head input is the
// NHWC bf16 output of dconv_last, [pix][64] with a row stride of ldx elements.
//
// All these kernels are HBM-bound (the head input alone is 128 B per pixel, the planes 4K B).  The conv kernels run
// on warp MMAs (mma.sync m16n8k16, bf16 in, fp32 accumulate) with the operands read straight from global memory into
// fragments: the reduction axis of an MMA may be permuted freely as long as A and B agree, and so may the columns
// of the result, so each kernel picks the permutation under which every lane loads and stores whole 16-byte vectors.
// The fp32 output gradients enter the MMAs as a hi + lo pair of bf16 values (two MMAs), which keeps their
// contribution to ~2^-17 relative: the weight gradient sums a million products and must not inherit bf16 rounding.
#include <algorithm>

#include "common.h"
#include "mma_sync.cuh"
#include "ptx.cuh"

namespace gap {

typedef __nv_bfloat16 bf16;

constexpr int kHeadC = 64;      // input channels of conv_last
constexpr int kMaxClasses = 16;  // one MMA M (or K) extent

// plane index of (class c, flat pixel p) in [n][K][hw]
__device__ __forceinline__ long long plane_idx(long long p, int c, int k, long long hw) {
  const long long img = p / hw;
  return p + (img * (k - 1) + c) * hw;
}

__device__ __forceinline__ uint32_t w_pair(const float* __restrict__ w, int k, int cls, int ch) {
  // two consecutive input channels of class row `cls` of the fp32 master, rounded to bf16 (0 for padding rows)
  return cls < k ? pack_bf16x2(__ldg(w + cls * kHeadC + ch), __ldg(w + cls * kHeadC + ch + 1)) : 0u;
}

__device__ __forceinline__ uint32_t w_col_pair(const float* __restrict__ w, int k, int c0, int ch) {
  // classes c0 and c0 + 1 of input channel ch
  const float a = c0 < k ? __ldg(w + c0 * kHeadC + ch) : 0.f;
  const float b = c0 + 1 < k ? __ldg(w + (c0 + 1) * kHeadC + ch) : 0.f;
  return pack_bf16x2(a, b);
}

// v = hi + lo with hi = bf16(v), lo = bf16(v - hi): two bf16x2 words for the value pair (v0, v1)
__device__ __forceinline__ void split_pair(float v0, float v1, uint32_t& hi, uint32_t& lo) {
  hi = pack_bf16x2(v0, v1);
  lo = pack_bf16x2(v0 - bf16_lo(hi), v1 - bf16_hi(hi));
}

// torch.argmax order: NaN above everything (the first NaN wins), ties to the lower index
__device__ __forceinline__ bool am_better(float v, int i, float bv, int bi) {
  const bool vn = v != v, bn = bv != bv;
  if (vn != bn) return vn;
  if (vn) return i < bi;
  return v > bv || (v == bv && i < bi);
}

// ------------------------------------------------------------------------------------------------
// Forward: out[c][pix] = bias[c] + sum_ch w[c][ch] * x[pix][ch]  as  D^T = W (16 classes x 64) * X^T (64 x 8 pixels).
// B fragment column = pixel g = lane/4 of an 8-pixel group; the lane loads channels q*16 .. q*16+15 of that pixel
// (q = lane%4, two 16-byte loads) and k-step s uses its words 2s (logical k 2q, 2q+1) and 2s+1 (logical 2q+8, 2q+9),
// i.e. logical k of step s maps to channel q*16 + s*4 + {0,1 | 2,3}; the weight fragments use the same map.
// Result: lane (g, q) holds classes g and g+8 of pixels 2q, 2q+1 of the group.  A warp works on 4 groups at a time.
// ------------------------------------------------------------------------------------------------
constexpr int kFwdGroups = 4;

__global__ void __launch_bounds__(256) conv1x1_ck_fwd_kernel(const bf16* __restrict__ x, long long ldx,
                                                             const float* __restrict__ w, const float* __restrict__ bias,
                                                             int k, long long hw, long long npix,
                                                             float* __restrict__ out, uint8_t* __restrict__ pred) {
  const int lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;
  uint32_t a[4][4];
#pragma unroll
  for (int s = 0; s < 4; ++s) {
    const int ch = q * 16 + s * 4;
    a[s][0] = w_pair(w, k, g, ch);
    a[s][1] = w_pair(w, k, g + 8, ch);
    a[s][2] = w_pair(w, k, g, ch + 2);
    a[s][3] = w_pair(w, k, g + 8, ch + 2);
  }
  const float b_lo = g < k ? __ldg(bias + g) : 0.f, b_hi = g + 8 < k ? __ldg(bias + g + 8) : 0.f;
  const long long groups = (npix + 7) >> 3;
  const long long warp0 = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5;
  const long long nwarps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  for (long long g0 = warp0 * kFwdGroups; g0 < groups; g0 += nwarps * kFwdGroups) {
    uint4 v[kFwdGroups][2];
#pragma unroll
    for (int u = 0; u < kFwdGroups; ++u) {
      const long long p = (g0 + u) * 8 + g;
      if (p < npix) {
        const uint4* src = reinterpret_cast<const uint4*>(x + p * ldx + q * 16);
        v[u][0] = __ldg(src);
        v[u][1] = __ldg(src + 1);
      } else {
        v[u][0] = v[u][1] = make_uint4(0u, 0u, 0u, 0u);
      }
    }
#pragma unroll
    for (int u = 0; u < kFwdGroups; ++u) {
      const uint32_t wd[8] = {v[u][0].x, v[u][0].y, v[u][0].z, v[u][0].w, v[u][1].x, v[u][1].y, v[u][1].z, v[u][1].w};
      float d[4] = {b_lo, b_lo, b_hi, b_hi};
#pragma unroll
      for (int s = 0; s < 4; ++s) mma_bf16_16816(d, a[s], wd[2 * s], wd[2 * s + 1]);
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const long long p = (g0 + u) * 8 + 2 * q + e;
        const bool ok = p < npix;
        if (ok) {
          const long long base = plane_idx(p, 0, k, hw);
          if (g < k) out[base + g * hw] = d[e];
          if (g + 8 < k) out[base + (g + 8) * hw] = d[2 + e];
        }
        if (pred != nullptr) {
          float bv = g < k ? d[e] : -INFINITY;
          int bi = g < k ? g : 64;
          if (g + 8 < k && am_better(d[2 + e], g + 8, bv, bi)) {
            bv = d[2 + e];
            bi = g + 8;
          }
#pragma unroll
          for (int o = 4; o < 32; o <<= 1) {       // the 8 lanes with the same q hold the other classes
            const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (am_better(ov, oi, bv, bi)) {
              bv = ov;
              bi = oi;
            }
          }
          if (ok && g == 0) pred[p] = static_cast<uint8_t>(bi);
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Input gradient: gx[pix][ch] = sum_c dl[c][pix] * w[c][ch]  as  D = dl^T (16 pixels x 16 classes) * W (16 x 8 ch).
// Result columns are permuted so that lane q ends with channels q*16 .. q*16+15 of its two pixel rows: n-tile t,
// column nn -> channel (nn/2)*16 + t*2 + nn%2; the rows then leave as two 16-byte stores each.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) conv1x1_ck_dgrad_kernel(const float* __restrict__ dl, const float* __restrict__ w,
                                                               int k, long long hw, long long npix,
                                                               bf16* __restrict__ gx, long long ldg) {
  const int lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;
  uint32_t b[8][2];
#pragma unroll
  for (int t = 0; t < 8; ++t) {
    const int ch = (g >> 1) * 16 + t * 2 + (g & 1);
    b[t][0] = w_col_pair(w, k, 2 * q, ch);
    b[t][1] = w_col_pair(w, k, 2 * q + 8, ch);
  }
  const long long tiles = (npix + 15) >> 4;
  const long long warp0 = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5;
  const long long nwarps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  for (long long tile = warp0; tile < tiles; tile += nwarps) {
    const long long p0 = tile * 16 + g, p1 = p0 + 8;
    float v[2][4];      // [row][class 2q, 2q+1, 2q+8, 2q+9]
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const long long p = r ? p1 : p0;
      const long long base = p < npix ? plane_idx(p, 0, k, hw) : 0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = 2 * q + (j & 1) + (j >> 1) * 8;
        v[r][j] = (p < npix && c < k) ? __ldg(dl + base + c * hw) : 0.f;
      }
    }
    uint32_t ahi[4], alo[4];
    split_pair(v[0][0], v[0][1], ahi[0], alo[0]);
    split_pair(v[1][0], v[1][1], ahi[1], alo[1]);
    split_pair(v[0][2], v[0][3], ahi[2], alo[2]);
    split_pair(v[1][2], v[1][3], ahi[3], alo[3]);
    uint32_t r0[8], r1[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      float d[4] = {0.f, 0.f, 0.f, 0.f};
      mma_bf16_16816(d, ahi, b[t][0], b[t][1]);
      mma_bf16_16816(d, alo, b[t][0], b[t][1]);
      r0[t] = pack_bf16x2(d[0], d[1]);
      r1[t] = pack_bf16x2(d[2], d[3]);
    }
    if (p0 < npix) {
      uint4* dst = reinterpret_cast<uint4*>(gx + p0 * ldg + q * 16);
      dst[0] = make_uint4(r0[0], r0[1], r0[2], r0[3]);
      dst[1] = make_uint4(r0[4], r0[5], r0[6], r0[7]);
    }
    if (p1 < npix) {
      uint4* dst = reinterpret_cast<uint4*>(gx + p1 * ldg + q * 16);
      dst[0] = make_uint4(r1[0], r1[1], r1[2], r1[3]);
      dst[1] = make_uint4(r1[4], r1[5], r1[6], r1[7]);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Weight gradient: dw[c][ch] += sum_pix dl[c][pix] * x[pix][ch]  as  D = dl (16 classes x 16 pixels) * X (16 x 8 ch).
// Reduction axis: lane q's logical k {2q, 2q+1, 2q+8, 2q+9} are pixels q*4 + {0,1,2,3} of the 16-pixel step.
// Columns: n-tile t, column nn -> channel nn*8 + t, so lane g loads channels g*8 .. g*8+7 (one 16-byte vector) of
// each of its four pixels and pairs them across pixels with byte permutes.  A CTA covers a contiguous pixel range,
// its warps stride through it; the partial sums meet in shared memory and leave with one atomic per (class, ch).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) conv1x1_ck_wgrad_kernel(const float* __restrict__ dl, const bf16* __restrict__ x,
                                                               long long ldx, int k, long long hw, long long npix,
                                                               long long per_cta, float* __restrict__ dw,
                                                               float* __restrict__ db) {
  __shared__ float red[kMaxClasses * kHeadC];
  __shared__ float redb[kMaxClasses];
  for (int i = threadIdx.x; i < kMaxClasses * kHeadC; i += blockDim.x) red[i] = 0.f;
  if (threadIdx.x < kMaxClasses) redb[threadIdx.x] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3, warp = threadIdx.x >> 5;
  const long long begin = blockIdx.x * per_cta;
  const long long end = std::min(npix, begin + per_cta);
  float acc[8][4];
#pragma unroll
  for (int t = 0; t < 8; ++t) acc[t][0] = acc[t][1] = acc[t][2] = acc[t][3] = 0.f;
  float bsum_lo = 0.f, bsum_hi = 0.f;
  for (long long s0 = begin + warp * 16; s0 < end; s0 += (blockDim.x >> 5) * 16) {
    uint4 xv[4];
    float dlo[4], dhi[4];      // classes g and g + 8 at the lane's four pixels
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const long long p = s0 + q * 4 + i;
      if (p < end) {
        xv[i] = __ldg(reinterpret_cast<const uint4*>(x + p * ldx + g * 8));
        const long long base = plane_idx(p, 0, k, hw);
        dlo[i] = g < k ? __ldg(dl + base + g * hw) : 0.f;
        dhi[i] = g + 8 < k ? __ldg(dl + base + (g + 8) * hw) : 0.f;
      } else {
        xv[i] = make_uint4(0u, 0u, 0u, 0u);
        dlo[i] = dhi[i] = 0.f;
      }
    }
    bsum_lo += (dlo[0] + dlo[1]) + (dlo[2] + dlo[3]);
    bsum_hi += (dhi[0] + dhi[1]) + (dhi[2] + dhi[3]);
    uint32_t ahi[4], alo[4];
    split_pair(dlo[0], dlo[1], ahi[0], alo[0]);
    split_pair(dhi[0], dhi[1], ahi[1], alo[1]);
    split_pair(dlo[2], dlo[3], ahi[2], alo[2]);
    split_pair(dhi[2], dhi[3], ahi[3], alo[3]);
    const uint32_t w0[4] = {xv[0].x, xv[0].y, xv[0].z, xv[0].w}, w1[4] = {xv[1].x, xv[1].y, xv[1].z, xv[1].w};
    const uint32_t w2[4] = {xv[2].x, xv[2].y, xv[2].z, xv[2].w}, w3[4] = {xv[3].x, xv[3].y, xv[3].z, xv[3].w};
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const uint32_t sel = (t & 1) ? 0x7632u : 0x5410u;     // high / low bf16 halves of word t/2
      const uint32_t b0 = __byte_perm(w0[t >> 1], w1[t >> 1], sel);
      const uint32_t b1 = __byte_perm(w2[t >> 1], w3[t >> 1], sel);
      mma_bf16_16816(acc[t], ahi, b0, b1);
      mma_bf16_16816(acc[t], alo, b0, b1);
    }
  }
  // acc[t] = {class g: ch (2q)*8+t, (2q+1)*8+t;  class g+8: same channels}
#pragma unroll
  for (int t = 0; t < 8; ++t) {
    atomicAdd(&red[g * kHeadC + (2 * q) * 8 + t], acc[t][0]);
    atomicAdd(&red[g * kHeadC + (2 * q + 1) * 8 + t], acc[t][1]);
    atomicAdd(&red[(g + 8) * kHeadC + (2 * q) * 8 + t], acc[t][2]);
    atomicAdd(&red[(g + 8) * kHeadC + (2 * q + 1) * 8 + t], acc[t][3]);
  }
  bsum_lo += __shfl_xor_sync(0xffffffffu, bsum_lo, 1);
  bsum_lo += __shfl_xor_sync(0xffffffffu, bsum_lo, 2);
  bsum_hi += __shfl_xor_sync(0xffffffffu, bsum_hi, 1);
  bsum_hi += __shfl_xor_sync(0xffffffffu, bsum_hi, 2);
  if (q == 0) {
    atomicAdd(&redb[g], bsum_lo);
    atomicAdd(&redb[g + 8], bsum_hi);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < k * kHeadC; i += blockDim.x) atomicAdd(dw + i, red[i]);
  if (db != nullptr && threadIdx.x < k) atomicAdd(db + threadIdx.x, redb[threadIdx.x]);
}

// ------------------------------------------------------------------------------------------------
// nn.CrossEntropyLoss(weight, ignore_index, reduction="mean") over the K planes against int64 labels [n][hw]:
//   loss = sum_i w[y_i] * (logsumexp(x_i) - x_i[y_i]) / sum_i w[y_i]   over pixels with y_i != ignore_index
//   grad[c][i] = grad_scale * w[y_i] / sum w * (softmax(x_i)[c] - [c == y_i])
// Pass 1 reads the labels only: sums[1] = sum w[y] and the count of labels outside [0, K) that are not ignore_index
// (they contribute nothing: no trap, a device assert would be a GPU fault).  Pass 2 reads the planes once, writes
// the gradient with the device-side 1 / sums[1] and accumulates sums[0]; a one-thread pass forms the loss.
// Sums are fp64 (0 / 0 = NaN when every pixel is ignored, as in torch).
// ------------------------------------------------------------------------------------------------
struct CeArgs {
  const float* x;
  const long long* labels;
  const float* weight;     // [K] or NULL
  long long ignore;
  int k;
  long long hw, npix;
  double* sums;            // [2]: sum w*nll, sum w
  long long* bad;          // += out-of-range labels
  float* grad;             // may be NULL
  float grad_scale;
  double* loss;
};

__device__ __forceinline__ void block_sum_d(double* dst, double v) {
  __shared__ double red[32];
  v = warp_sum_d(v);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  if (wid == 0) {
    double t = lane < static_cast<int>((blockDim.x + 31) >> 5) ? red[lane] : 0.0;
    t = warp_sum_d(t);
    if (lane == 0 && t != 0.0) atomicAdd(dst, t);
  }
}

__global__ void ce_zero_kernel(double* sums) {
  if (threadIdx.x < 2) sums[threadIdx.x] = 0.0;
}

__global__ void __launch_bounds__(256) ce_labels_kernel(const CeArgs a) {
  double wsum = 0.0;
  unsigned int nbad = 0;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < a.npix;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long y = a.labels[i];
    if (y == a.ignore) continue;
    if (y < 0 || y >= a.k) {
      ++nbad;
      continue;
    }
    wsum += a.weight ? static_cast<double>(__ldg(a.weight + y)) : 1.0;
  }
  block_sum_d(a.sums + 1, wsum);
  for (int o = 16; o > 0; o >>= 1) nbad += __shfl_xor_sync(0xffffffffu, nbad, o);
  if ((threadIdx.x & 31) == 0 && nbad) atomicAdd(reinterpret_cast<unsigned long long*>(a.bad), nbad);
}

template <int K>
__global__ void __launch_bounds__(256) ce_main_kernel(const CeArgs a) {
  const int k = K > 0 ? K : a.k;
  const float inv_w = static_cast<float>(1.0 / a.sums[1]);
  double lsum = 0.0;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < a.npix;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long img = i / a.hw;
    const long long base = i + img * (k - 1) * a.hw;
    const long long y = a.labels[i];
    const bool valid = y != a.ignore && y >= 0 && y < k;
    float v[kMaxClasses];
    float m = -INFINITY, xy = 0.f;
#pragma unroll
    for (int c = 0; c < kMaxClasses; ++c) {
      if (c < k) {
        v[c] = a.x[base + c * a.hw];
        m = fmaxf(m, v[c]);
        if (c == y) xy = v[c];
      }
    }
    float se = 0.f;
#pragma unroll
    for (int c = 0; c < kMaxClasses; ++c) {
      if (c < k) {
        v[c] = expf(v[c] - m);       // v now holds exp(x - max); the logit itself is kept as xy below
        se += v[c];
      }
    }
    const float lse = m + logf(se);
    const int yc = valid ? static_cast<int>(y) : 0;
    const float wy = valid ? (a.weight ? __ldg(a.weight + yc) : 1.f) : 0.f;
    if (valid) {
      lsum += static_cast<double>(wy) * static_cast<double>(lse - xy);
    }
    if (a.grad != nullptr) {
      const float f = a.grad_scale * wy * inv_w;
      const float inv_se = 1.f / se;
#pragma unroll
      for (int c = 0; c < kMaxClasses; ++c) {
        if (c < k) {
          const float p = v[c] * inv_se;
          a.grad[base + c * a.hw] = valid ? f * (p - (c == yc ? 1.f : 0.f)) : 0.f;
        }
      }
    }
  }
  block_sum_d(a.sums, lsum);
}

__global__ void ce_finish_kernel(const CeArgs a) {
  if (threadIdx.x == 0) a.loss[0] = a.sums[0] / a.sums[1];
}

// ------------------------------------------------------------------------------------------------
// Softmax point term + multi-class Dice over the K planes, p = softmax(x), V = pixels with y != ignore, 0 <= y < K:
//   loss = w_point * Point + (1 - w_point) * Dice,   Dice = 1 - 1/(K-1) sum_{k>=1} (2 I_k + s) / (P_k + T_k + s)
//   I_k = sum_V p_k [y=k], P_k = sum_V p_k, T_k = sum_V [y=k]  (whole batch; class 0 is not a Dice class)
//   mode 0: Point = sum_V w[y] (-log p_y) / sum_V w[y]                   (nn.CrossEntropyLoss(weight, ignore_index))
//   mode 1: Point = sum_V a[y] (1 - p_y)^gamma (-log p_y) / |V|          (softmax focal loss, a = class_weight)
// Pass 1 (stats) reads planes and labels once and accumulates the fp64 sums [num, norm, I_1.., P_1.., T_1..]
// (3(K-1)+2 of them) and the out-of-range label count; pass 2 derives the per-class Dice coefficients from the sums in
// every CTA (no finalize launch, no host sync), recomputes the softmax and writes the gradient; block 0 writes the loss.
// ------------------------------------------------------------------------------------------------
constexpr int kDiceSums = 3 * (kMaxClasses - 1) + 2;

struct DiceArgs {
  const float* x;
  const long long* labels;
  const float* weight;     // [K] or NULL (all 1)
  long long ignore;
  int k, mode;
  long long hw, npix;
  float w_point, gamma, smooth;
  double* sums;            // [3(K-1)+2]
  long long* bad;          // += out-of-range labels
  float* grad;             // may be NULL
  float grad_scale;
  double* loss;
};

// (1 - q)^gamma (-log q) and its log-ratio helper for the focal term, from r = sum_{c != y} p_c (accurate for confident
// pixels, where 1 - q cancels) and nll_lse = lse - x_y (accurate for unlikely labels, where log1p(-r) rounds)
__device__ __forceinline__ float focal_nll(float r, float nll_lse) { return r < 0.5f ? -log1pf(-r) : nll_lse; }
__device__ __forceinline__ float focal_logq_over_r(float r, float nll_lse) {   // log(q) / r, -> -1 at r = 0
  return r == 0.f ? -1.f : (r < 0.5f ? log1pf(-r) / r : -nll_lse / r);
}
__device__ __forceinline__ float pow_gamma(float r, float gamma) { return gamma == 2.f ? r * r : powf(r, gamma); }

template <int K>
__global__ void __launch_bounds__(256) dice_stats_kernel(const DiceArgs a) {
  const int k = K > 0 ? K : a.k;
  float I[kMaxClasses], P[kMaxClasses], T[kMaxClasses];
#pragma unroll
  for (int c = 0; c < kMaxClasses; ++c) I[c] = P[c] = T[c] = 0.f;
  float num = 0.f, norm = 0.f;
  unsigned int nbad = 0;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < a.npix;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long y = a.labels[i];
    if (y == a.ignore) continue;
    if (y < 0 || y >= k) {
      ++nbad;
      continue;
    }
    const long long base = i + (i / a.hw) * (k - 1) * a.hw;
    float v[kMaxClasses];
    float m = -INFINITY, xy = 0.f;
#pragma unroll
    for (int c = 0; c < kMaxClasses; ++c) {
      if (c < k) {
        v[c] = a.x[base + c * a.hw];
        m = fmaxf(m, v[c]);
        if (c == y) xy = v[c];
      }
    }
    float se = 0.f;
#pragma unroll
    for (int c = 0; c < kMaxClasses; ++c) {
      if (c < k) {
        v[c] = expf(v[c] - m);
        se += v[c];
      }
    }
    const float inv_se = 1.f / se;
    float r = 0.f;
#pragma unroll
    for (int c = 0; c < kMaxClasses; ++c) {
      if (c < k) {
        const float p = v[c] * inv_se;
        P[c] += p;
        if (c == y) {
          I[c] += p;
          T[c] += 1.f;
        } else {
          r += p;
        }
      }
    }
    const float nll_lse = m + logf(se) - xy;
    const float wy = a.weight ? __ldg(a.weight + y) : 1.f;
    if (a.mode == 0) {
      num += wy * nll_lse;
      norm += wy;
    } else {
      num += wy * pow_gamma(r, a.gamma) * focal_nll(r, nll_lse);
      norm += 1.f;
    }
  }
  // CTA reduction in fp64: warp shuffles, then one slot per (sum, warp) in shared memory, one atomic per sum
  __shared__ double red[kDiceSums][8];
  __shared__ unsigned int red_bad[8];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int nsum = 3 * (k - 1) + 2;
  auto put = [&](int s, float v) {
    const double d = warp_sum_d(static_cast<double>(v));
    if (lane == 0) red[s][wid] = d;
  };
  put(0, num);
  put(1, norm);
#pragma unroll
  for (int c = 1; c < kMaxClasses; ++c) {
    if (c < k) {
      put(1 + c, I[c]);
      put(k + c, P[c]);
      put(2 * k - 1 + c, T[c]);
    }
  }
  for (int o = 16; o > 0; o >>= 1) nbad += __shfl_xor_sync(0xffffffffu, nbad, o);
  if (lane == 0) red_bad[wid] = nbad;
  __syncthreads();
  const int nw = blockDim.x >> 5;
  for (int s = threadIdx.x; s < nsum; s += blockDim.x) {
    double t = 0.0;
    for (int w = 0; w < nw; ++w) t += red[s][w];
    if (t != 0.0) atomicAdd(a.sums + s, t);
  }
  if (threadIdx.x == 0) {
    unsigned long long b = 0;
    for (int w = 0; w < nw; ++w) b += red_bad[w];
    if (b) atomicAdd(reinterpret_cast<unsigned long long*>(a.bad), b);
  }
}

template <int K>
__global__ void __launch_bounds__(256) dice_grad_kernel(const DiceArgs a) {
  const int k = K > 0 ? K : a.k;
  // g_c = A_c [y=c] + B_c is d(Dice)/d(p_c) at a counted pixel (A_0 = B_0 = 0)
  __shared__ float sA[kMaxClasses], sB[kMaxClasses];
  __shared__ float s_inv_norm;
  const double* S = a.sums;
  if (threadIdx.x < kMaxClasses) {
    const int c = threadIdx.x;
    float A = 0.f, B = 0.f;
    if (c >= 1 && c < k) {
      const double U = S[k + c] + S[2 * k - 1 + c] + a.smooth;
      A = static_cast<float>(-2.0 / ((k - 1) * U));
      B = static_cast<float>((2.0 * S[1 + c] + a.smooth) / ((k - 1) * U * U));
    }
    sA[c] = A;
    sB[c] = B;
  }
  if (threadIdx.x == 0) {
    s_inv_norm = static_cast<float>(1.0 / S[1]);
    if (blockIdx.x == 0) {
      double ratio = 0.0;
      for (int c = 1; c < k; ++c) ratio += (2.0 * S[1 + c] + a.smooth) / (S[k + c] + S[2 * k - 1 + c] + a.smooth);
      const double dice = 1.0 - ratio / (k - 1);
      a.loss[0] = a.w_point * (S[0] / S[1]) + (1.0 - a.w_point) * dice;
    }
  }
  if (a.grad == nullptr) return;
  __syncthreads();
  float A[kMaxClasses], B[kMaxClasses];
#pragma unroll
  for (int c = 0; c < kMaxClasses; ++c) {
    A[c] = c < k ? sA[c] : 0.f;
    B[c] = c < k ? sB[c] : 0.f;
  }
  const float inv_norm = s_inv_norm;
  const float wp = a.grad_scale * a.w_point, wd = a.grad_scale * (1.f - a.w_point);
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < a.npix;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long base = i + (i / a.hw) * (k - 1) * a.hw;
    const long long y = a.labels[i];
    if (y == a.ignore || y < 0 || y >= k) {
#pragma unroll
      for (int c = 0; c < kMaxClasses; ++c)
        if (c < k) a.grad[base + c * a.hw] = 0.f;
      continue;
    }
    float v[kMaxClasses];
    float m = -INFINITY, xy = 0.f;
#pragma unroll
    for (int c = 0; c < kMaxClasses; ++c) {
      if (c < k) {
        v[c] = a.x[base + c * a.hw];
        m = fmaxf(m, v[c]);
        if (c == y) xy = v[c];
      }
    }
    float se = 0.f;
#pragma unroll
    for (int c = 0; c < kMaxClasses; ++c) {
      if (c < k) {
        v[c] = expf(v[c] - m);
        se += v[c];
      }
    }
    const float inv_se = 1.f / se;
    float sg = 0.f, r = 0.f, q = 0.f;
#pragma unroll
    for (int c = 0; c < kMaxClasses; ++c) {
      if (c < k) {
        v[c] *= inv_se;                    // v now holds p
        sg += v[c] * ((c == y ? A[c] : 0.f) + B[c]);
        if (c == y) q = v[c];
        else r += v[c];
      }
    }
    const float wy = a.weight ? __ldg(a.weight + y) : 1.f;
    // point term: d/dx_c = fp * (p_c - [c=y])
    float fp;
    if (a.mode == 0) {
      fp = wy * inv_norm;
    } else {
      const float nll_lse = m + logf(se) - xy;
      fp = -wy * pow_gamma(r, a.gamma) * (a.gamma * q * focal_logq_over_r(r, nll_lse) - 1.f) * inv_norm;
    }
#pragma unroll
    for (int c = 0; c < kMaxClasses; ++c) {
      if (c < k) {
        const float g = (c == y ? A[c] : 0.f) + B[c];
        const float dpoint = fp * (v[c] - (c == y ? 1.f : 0.f));
        const float ddice = v[c] * (g - sg);
        a.grad[base + c * a.hw] = wp * dpoint + wd * ddice;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Per-sample K x K confusion matrix: counts[n][label][argmax_c logits[n][c][pix]] += 1 over pixels whose label is in
// [0, K) (ignore_index and out-of-range labels are skipped).  gridDim.y = samples; a warp adds equal bins once
// (__match_any_sync), shared-memory histograms, one 64-bit atomic per non-empty bin and CTA.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) confusion_ck_kernel(const float* __restrict__ logits,
                                                           const long long* __restrict__ labels, int k, long long hw,
                                                           long long ignore, unsigned long long* __restrict__ counts) {
  __shared__ unsigned int hist[kMaxClasses * kMaxClasses];
  for (int i = threadIdx.x; i < k * k; i += blockDim.x) hist[i] = 0u;
  __syncthreads();
  const long long img = blockIdx.y;
  const float* xs = logits + img * k * hw;
  const long long* ys = labels + img * hw;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i0 = blockIdx.x * static_cast<long long>(blockDim.x); i0 < hw; i0 += stride) {   // uniform per warp
    const long long i = i0 + threadIdx.x;
    int bin = -1;
    if (i < hw) {
      const long long y = ys[i];
      if (y != ignore && y >= 0 && y < k) {
        float bv = xs[i];
        int bi = 0;
        for (int c = 1; c < k; ++c) {
          const float v = xs[c * hw + i];
          if (am_better(v, c, bv, bi)) {
            bv = v;
            bi = c;
          }
        }
        bin = static_cast<int>(y) * k + bi;
      }
    }
    const unsigned int peers = __match_any_sync(0xffffffffu, bin);
    if (bin >= 0 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&hist[bin], __popc(peers));
  }
  __syncthreads();
  for (int i = threadIdx.x; i < k * k; i += blockDim.x)
    if (hist[i]) atomicAdd(counts + img * k * k + i, static_cast<unsigned long long>(hist[i]));
}

static inline int ck_grid(long long work, int block, int max_blocks) {
  long long g = (work + block - 1) / block;
  if (g < 1) g = 1;
  return static_cast<int>(g < max_blocks ? g : max_blocks);
}

}  // namespace gap

using namespace gap;

#define CK_LAUNCH_OK()            \
  do {                            \
    GAP_CUDA(cudaGetLastError()); \
    return 0;                     \
  } while (0)

extern "C" {

int gap_conv1x1_ck_fwd(const void* x, int64_t ldx, const float* w, const float* bias, int k, int n, int64_t hw,
                       float* out, uint8_t* pred, void* stream) {
  GAP_CHECK_ARG(k >= 1 && k <= kMaxClasses, "gap_conv1x1_ck_fwd: k must be 1..16, got %d", k);
  GAP_CHECK_ARG(x && w && bias && out && n > 0 && hw > 0 && ldx >= kHeadC && ldx % 8 == 0,
                "gap_conv1x1_ck_fwd: bad arguments");
  const long long npix = static_cast<long long>(n) * hw;
  const long long warps = ((npix + 7) / 8 + kFwdGroups - 1) / kFwdGroups;
  conv1x1_ck_fwd_kernel<<<ck_grid(warps * 32, 256, 148 * 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const bf16*>(x), ldx, w, bias, k, hw, npix, out, pred);
  CK_LAUNCH_OK();
}

int gap_conv1x1_ck_dgrad(const float* dl, const float* w, int k, int n, int64_t hw, void* gx, int64_t ldg, void* stream) {
  GAP_CHECK_ARG(k >= 1 && k <= kMaxClasses, "gap_conv1x1_ck_dgrad: k must be 1..16, got %d", k);
  GAP_CHECK_ARG(dl && w && gx && n > 0 && hw > 0 && ldg >= kHeadC && ldg % 8 == 0, "gap_conv1x1_ck_dgrad: bad arguments");
  const long long npix = static_cast<long long>(n) * hw;
  conv1x1_ck_dgrad_kernel<<<ck_grid((npix + 15) / 16 * 32, 256, 148 * 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      dl, w, k, hw, npix, static_cast<bf16*>(gx), ldg);
  CK_LAUNCH_OK();
}

int gap_conv1x1_ck_wgrad(const float* dl, const void* x, int64_t ldx, int k, int n, int64_t hw, float* dw, float* db,
                         void* stream) {
  GAP_CHECK_ARG(k >= 1 && k <= kMaxClasses, "gap_conv1x1_ck_wgrad: k must be 1..16, got %d", k);
  GAP_CHECK_ARG(dl && x && dw && n > 0 && hw > 0 && ldx >= kHeadC && ldx % 8 == 0, "gap_conv1x1_ck_wgrad: bad arguments");
  const long long npix = static_cast<long long>(n) * hw;
  const int grid = ck_grid(npix, 8 * 16 * 4, 148 * 2);           // >= 4 steps of 16 pixels per warp
  const long long per_cta = ((npix + grid - 1) / grid + 15) / 16 * 16;
  conv1x1_ck_wgrad_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(dl, static_cast<const bf16*>(x), ldx, k,
                                                                               hw, npix, per_cta, dw, db);
  CK_LAUNCH_OK();
}

int gap_seg_ce_loss(const float* logits, const int64_t* labels, int k, int n, int64_t hw, const float* class_weight,
                    int64_t ignore_index, double* sums2, int64_t* bad_labels, float* grad, float grad_scale,
                    double* loss, void* stream) {
  GAP_CHECK_ARG(k >= 1 && k <= kMaxClasses, "gap_seg_ce_loss: k must be 1..16, got %d", k);
  GAP_CHECK_ARG(logits && labels && sums2 && bad_labels && loss && n > 0 && hw > 0, "gap_seg_ce_loss: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long npix = static_cast<long long>(n) * hw;
  CeArgs a{logits, reinterpret_cast<const long long*>(labels), class_weight, ignore_index, k, hw, npix, sums2,
           reinterpret_cast<long long*>(bad_labels), grad, grad_scale, loss};
  ce_zero_kernel<<<1, 32, 0, st>>>(sums2);
  ce_labels_kernel<<<ck_grid(npix, 256, 148 * 4), 256, 0, st>>>(a);
  const int grid = ck_grid(npix, 256, 148 * 8);
  switch (k) {     // the common small class counts get fully unrolled plane loops
    case 2: ce_main_kernel<2><<<grid, 256, 0, st>>>(a); break;
    case 3: ce_main_kernel<3><<<grid, 256, 0, st>>>(a); break;
    case 7: ce_main_kernel<7><<<grid, 256, 0, st>>>(a); break;
    default: ce_main_kernel<0><<<grid, 256, 0, st>>>(a); break;
  }
  GAP_CUDA(cudaGetLastError());
  ce_finish_kernel<<<1, 32, 0, st>>>(a);
  CK_LAUNCH_OK();
}

int gap_seg_softmax_dice(const float* logits, const int64_t* labels, int k, int n, int64_t hw, int mode, float w_point,
                         float gamma, float smooth, const float* class_weight, int64_t ignore_index, double* sums,
                         int64_t* bad_labels, float* grad, float grad_scale, double* loss, void* stream) {
  GAP_CHECK_ARG(k >= 2 && k <= kMaxClasses, "gap_seg_softmax_dice: k must be 2..16, got %d", k);
  GAP_CHECK_ARG(logits && labels && sums && bad_labels && loss && n > 0 && hw > 0 && (mode == 0 || mode == 1),
                "gap_seg_softmax_dice: bad arguments");
  GAP_CHECK_ARG(smooth > 0.f && gamma >= 0.f && w_point >= 0.f && w_point <= 1.f,
                "gap_seg_softmax_dice: need smooth > 0, gamma >= 0 and 0 <= w_point <= 1");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long npix = static_cast<long long>(n) * hw;
  DiceArgs a{logits, reinterpret_cast<const long long*>(labels), class_weight, ignore_index, k, mode, hw, npix,
             w_point, gamma, smooth, sums, reinterpret_cast<long long*>(bad_labels), grad, grad_scale, loss};
  GAP_CUDA(cudaMemsetAsync(sums, 0, sizeof(double) * (3 * (k - 1) + 2), st));
  const int gs = ck_grid(npix, 256, 148 * 4);
  const int gg = grad ? ck_grid(npix, 256, 148 * 8) : 1;      // without a gradient only block 0 (the loss) runs
  switch (k) {     // the common small class counts get fully unrolled plane loops
    case 2: dice_stats_kernel<2><<<gs, 256, 0, st>>>(a); dice_grad_kernel<2><<<gg, 256, 0, st>>>(a); break;
    case 3: dice_stats_kernel<3><<<gs, 256, 0, st>>>(a); dice_grad_kernel<3><<<gg, 256, 0, st>>>(a); break;
    case 7: dice_stats_kernel<7><<<gs, 256, 0, st>>>(a); dice_grad_kernel<7><<<gg, 256, 0, st>>>(a); break;
    default: dice_stats_kernel<0><<<gs, 256, 0, st>>>(a); dice_grad_kernel<0><<<gg, 256, 0, st>>>(a); break;
  }
  CK_LAUNCH_OK();
}

int gap_seg_confusion_ck(const float* logits, const int64_t* labels, int k, int n, int64_t hw, int64_t ignore_index,
                         int64_t* counts, void* stream) {
  GAP_CHECK_ARG(k >= 1 && k <= kMaxClasses, "gap_seg_confusion_ck: k must be 1..16, got %d", k);
  GAP_CHECK_ARG(logits && labels && counts && n > 0 && n < 65536 && hw > 0, "gap_seg_confusion_ck: bad arguments");
  const int bx = static_cast<int>(std::min<long long>((hw + 255) / 256, 148 * 8 / std::min(n, 148) + 1));
  dim3 grid(bx, n);
  confusion_ck_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      logits, reinterpret_cast<const long long*>(labels), k, hw, ignore_index,
      reinterpret_cast<unsigned long long*>(counts));
  CK_LAUNCH_OK();
}

}  // extern "C"
