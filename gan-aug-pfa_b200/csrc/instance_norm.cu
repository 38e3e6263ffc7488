// InstanceNorm2d(affine=False, track_running_stats=False) for the pix2pix `--norm instance` configuration
// (norm_layer=nn.InstanceNorm2d in UnetSkipConnectionBlock / NLayerDiscriminator): statistics per (image, channel) over
// H*W, in train and eval mode alike.
//
//   gap_in_stats       sums[0][n*C+c] += sum y,  sums[1][n*C+c] += sum y^2
//   (gap_bn_finalize with c = N*C, count = H*W and no gamma / beta / running buffers turns the sums into per-(n,c)
//    scale = invstd, shift = -mean*invstd, mean, invstd and re-zeroes them)
//   gap_in_act         out1 = act1(y*scale + shift), out2 = act2(same)
//   gap_in_bwd_reduce  d = (xhat > 0) ? g1 + g2 : slope*g1;  sums[0] += sum d,  sums[1] += sum d*xhat
//   gap_in_bwd_apply   dy = invstd * (d - sums[0]/hw - xhat*sums[1]/hw);  dbias[c] += sum over n, pixels of dy (fp32)
//
// Thread layout (as bn_act_slope_kernel / bn_bwd_kernel): threadIdx.x walks 8-channel (16-byte) groups, threadIdx.y
// walks pixels, U pixels in flight per thread.  Unlike the BatchNorm kernels every CTA covers a pixel range INSIDE ONE
// image (grid = (chunks, n)), so its per-(n,c) scale / shift / sums stay in registers for the whole CTA.
#include "common.h"
#include "ptx.cuh"

namespace gap {
namespace {

constexpr int kInU = 4;             // pixels in flight per thread
constexpr int kInMaxC = 2048;       // keeps the [by][C][2] fp32 reduction under the 48 KB static shared-memory limit

typedef __nv_bfloat16 bf16;

__device__ __forceinline__ void in_unpack(const uint4& raw, float (&v)[8]) {
  const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    v[2 * j] = bf16_lo(w[j]);
    v[2 * j + 1] = bf16_hi(w[j]);
  }
}

__device__ __forceinline__ void in_act8(const float (&v)[8], int act, uint32_t (&pk)[4]) {
  if (act == GAP_ACT_RELU) {
#pragma unroll
    for (int j = 0; j < 4; ++j) pk[j] = pack_bf16x2(fmaxf(v[2 * j], 0.f), fmaxf(v[2 * j + 1], 0.f));
  } else if (act == GAP_ACT_LRELU) {
#pragma unroll
    for (int j = 0; j < 4; ++j) pk[j] = pack_bf16x2(fmaxf(v[2 * j], 0.2f * v[2 * j]), fmaxf(v[2 * j + 1], 0.2f * v[2 * j + 1]));
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) pk[j] = pack_bf16x2(v[2 * j], v[2 * j + 1]);
  }
}

__device__ __forceinline__ void in_loadf8(const float* p, float (&v)[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

// CTA (blockIdx.x, img = blockIdx.y) covers pixels [p0, p1) of image img
__device__ __forceinline__ void in_range(long long hw, long long span, long long& p0, long long& p1) {
  p0 = static_cast<long long>(blockIdx.x) * span;
  p1 = p0 + span < hw ? p0 + span : hw;
}

// Block-wide sum of red[by][c*k] over by, one atomic per column: fp64 into sums[which*nc + img*c + ch] (k = 2) or fp32
// into dbias[ch] (k = 1).
__device__ __forceinline__ void in_flush(const float* red, int c, int k, double* sums, int nc, int img, float* dbias) {
  __syncthreads();
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  const int nthr = blockDim.x * blockDim.y;
  for (int i = tid; i < c * k; i += nthr) {
    double tot = 0.0;
    for (int r = 0; r < static_cast<int>(blockDim.y); ++r) tot += red[static_cast<size_t>(r) * c * k + i];
    if (dbias)
      atomicAdd(dbias + i, static_cast<float>(tot));
    else
      atomicAdd(sums + (i & 1) * nc + img * c + (i >> 1), tot);
  }
}

__global__ void __launch_bounds__(256) in_stats_kernel(const bf16* __restrict__ y, long long ld, long long hw, int c,
                                                       long long span, double* __restrict__ sums, int nc) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float in_red[];   // [blockDim.y][c][2]
  const int cv = c >> 3, img = blockIdx.y;
  long long p0, p1;
  in_range(hw, span, p0, p1);
  const bf16* base = y + static_cast<long long>(img) * hw * ld;
  const long long step = static_cast<long long>(kInU) * blockDim.y;
  for (int cg = threadIdx.x; cg < cv; cg += blockDim.x) {
    const int c8 = cg << 3;
    float s1[8] = {0, 0, 0, 0, 0, 0, 0, 0}, s2[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (long long pix0 = p0 + threadIdx.y; pix0 < p1; pix0 += step) {
      uint4 raw[kInU];
#pragma unroll
      for (int u = 0; u < kInU; ++u) {
        const long long pix = pix0 + u * static_cast<long long>(blockDim.y);
        if (pix < p1) raw[u] = __ldg(reinterpret_cast<const uint4*>(base + pix * ld + c8));
      }
#pragma unroll
      for (int u = 0; u < kInU; ++u) {
        if (pix0 + u * static_cast<long long>(blockDim.y) >= p1) break;
        float v[8];
        in_unpack(raw[u], v);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          s1[j] += v[j];
          s2[j] = fmaf(v[j], v[j], s2[j]);
        }
      }
    }
    float* slot = in_red + (static_cast<size_t>(threadIdx.y) * c + c8) * 2;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      slot[2 * j] = s1[j];
      slot[2 * j + 1] = s2[j];
    }
  }
  in_flush(in_red, c, 2, sums, nc, img, nullptr);
}

__global__ void __launch_bounds__(256, 2) in_act_kernel(const bf16* __restrict__ y, long long ld, long long hw, int c,
                                                        long long span, const float* __restrict__ scale,
                                                        const float* __restrict__ shift, bf16* __restrict__ o1,
                                                        long long ld1, int act1, bf16* __restrict__ o2, long long ld2,
                                                        int act2) {
  pdl_trigger();
  pdl_wait();
  const int cv = c >> 3, img = blockIdx.y;
  long long p0, p1;
  in_range(hw, span, p0, p1);
  const long long row0 = static_cast<long long>(img) * hw;
  const long long step = static_cast<long long>(kInU) * blockDim.y;
  for (int cg = threadIdx.x; cg < cv; cg += blockDim.x) {
    const int c8 = cg << 3;
    float sc[8], sh[8];
    in_loadf8(scale + img * c + c8, sc);
    in_loadf8(shift + img * c + c8, sh);
    for (long long pix0 = p0 + threadIdx.y; pix0 < p1; pix0 += step) {
      uint4 raw[kInU];
#pragma unroll
      for (int u = 0; u < kInU; ++u) {
        const long long pix = pix0 + u * static_cast<long long>(blockDim.y);
        if (pix < p1) raw[u] = __ldg(reinterpret_cast<const uint4*>(y + (row0 + pix) * ld + c8));
      }
#pragma unroll
      for (int u = 0; u < kInU; ++u) {
        const long long pix = pix0 + u * static_cast<long long>(blockDim.y);
        if (pix >= p1) break;
        float v[8];
        in_unpack(raw[u], v);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = fmaf(v[j], sc[j], sh[j]);
        uint32_t pk[4];
        in_act8(v, act1, pk);
        *reinterpret_cast<uint4*>(o1 + (row0 + pix) * ld1 + c8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        if (o2) {
          in_act8(v, act2, pk);
          *reinterpret_cast<uint4*>(o2 + (row0 + pix) * ld2 + c8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
      }
    }
  }
}

struct InBwdArgs {
  const bf16* y;
  long long ld_y;
  const bf16* g1;
  long long ld_g1;
  const bf16* g2;
  long long ld_g2;
  float slope;
  const float* scale;   // [N][C] = invstd (no affine)
  const float* shift;   // [N][C] = -mean * invstd
  long long hw;
  int c;
  int nc;
  long long span;
  double* sums;         // [2][N*C]
  double inv_hw;
  bf16* dy;
  long long ld_dy;
  float* dbias;
};

// APPLY = false: the reduce pass; true: the apply pass.  G2: a second gradient source (the ReLU'd U-Net skip copy).
template <bool APPLY, bool G2>
__global__ void __launch_bounds__(256, 2) in_bwd_kernel(const InBwdArgs a) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float in_red[];   // reduce: [blockDim.y][c][2]; apply with dbias: [blockDim.y][c]
  const int cv = a.c >> 3, img = blockIdx.y;
  long long p0, p1;
  in_range(a.hw, a.span, p0, p1);
  const long long row0 = static_cast<long long>(img) * a.hw;
  const long long step = static_cast<long long>(kInU) * blockDim.y;
  const bool do_bias = APPLY && a.dbias != nullptr;
  for (int cg = threadIdx.x; cg < cv; cg += blockDim.x) {
    const int c8 = cg << 3;
    const int nc0 = img * a.c + c8;
    // apply:  dy = sc*(d - m1 - xhat*m2) = sc*d + ca*y + cb,  xhat = y*sc + sh,  ca = -sc*sc*m2,  cb = -sc*(m1 + sh*m2)
    float sc[8], sh[8], ca[8], cb[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      sc[j] = a.scale[nc0 + j];
      sh[j] = a.shift[nc0 + j];
      ca[j] = cb[j] = 0.f;
      if (APPLY) {
        const float m1 = static_cast<float>(a.sums[nc0 + j] * a.inv_hw);
        const float m2 = static_cast<float>(a.sums[a.nc + nc0 + j] * a.inv_hw);
        ca[j] = -sc[j] * sc[j] * m2;
        cb[j] = -sc[j] * fmaf(sh[j], m2, m1);
      }
    }
    float s1[8] = {0, 0, 0, 0, 0, 0, 0, 0}, s2[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (long long pix0 = p0 + threadIdx.y; pix0 < p1; pix0 += step) {
      uint4 yr[kInU], g1r[kInU], g2r[G2 ? kInU : 1];
#pragma unroll
      for (int u = 0; u < kInU; ++u) {
        const long long pix = row0 + pix0 + u * static_cast<long long>(blockDim.y);
        if (pix0 + u * static_cast<long long>(blockDim.y) < p1) {
          yr[u] = __ldg(reinterpret_cast<const uint4*>(a.y + pix * a.ld_y + c8));
          g1r[u] = __ldg(reinterpret_cast<const uint4*>(a.g1 + pix * a.ld_g1 + c8));
          if (G2) g2r[u] = __ldg(reinterpret_cast<const uint4*>(a.g2 + pix * a.ld_g2 + c8));
        }
      }
#pragma unroll
      for (int u = 0; u < kInU; ++u) {
        if (pix0 + u * static_cast<long long>(blockDim.y) >= p1) break;
        const long long pix = row0 + pix0 + u * static_cast<long long>(blockDim.y);
        float yv[8], g1[8], g2[8];
        in_unpack(yr[u], yv);
        in_unpack(g1r[u], g1);
        if (G2) in_unpack(g2r[G2 ? u : 0], g2);
        float d[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float xh = fmaf(yv[j], sc[j], sh[j]);
          d[j] = xh > 0.f ? (G2 ? g1[j] + g2[j] : g1[j]) : a.slope * g1[j];
          if (!APPLY) {
            s1[j] += d[j];
            s2[j] = fmaf(d[j], xh, s2[j]);
          }
        }
        if (APPLY) {
          float o[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            o[j] = fmaf(sc[j], d[j], fmaf(ca[j], yv[j], cb[j]));
            s1[j] += o[j];
          }
          uint32_t pk[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) pk[j] = pack_bf16x2(o[2 * j], o[2 * j + 1]);
          *reinterpret_cast<uint4*>(a.dy + pix * a.ld_dy + c8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
      }
    }
    if (!APPLY) {
      float* slot = in_red + (static_cast<size_t>(threadIdx.y) * a.c + c8) * 2;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        slot[2 * j] = s1[j];
        slot[2 * j + 1] = s2[j];
      }
    } else if (do_bias) {
      float* slot = in_red + static_cast<size_t>(threadIdx.y) * a.c + c8;
#pragma unroll
      for (int j = 0; j < 8; ++j) slot[j] = s1[j];
    }
  }
  if (!APPLY)
    in_flush(in_red, a.c, 2, a.sums, a.nc, img, nullptr);
  else if (do_bias)
    in_flush(in_red, a.c, 1, nullptr, 0, img, a.dbias);
}

// Launch geometry: blockDim (bx 8-channel groups, by pixel rows); grid (chunks, n) with `span` pixels per CTA.  About four
// CTAs per SM in all, and at least kInU pixel rows per CTA (the 2x2 / 4x4 maps of the U-Net bottleneck get one CTA per image).
struct InGeom {
  dim3 grid, block;
  long long span;
};

InGeom in_geom(int n, long long hw, int c) {
  const int cv = c / 8;
  const int bx = cv < 128 ? cv : 128;
  const int by = 256 / bx < 1 ? 1 : 256 / bx;
  const long long want = (4LL * sm_count() + n - 1) / n;
  const long long most = (hw + static_cast<long long>(by) * kInU - 1) / (static_cast<long long>(by) * kInU);
  long long chunks = want < most ? want : most;
  if (chunks < 1) chunks = 1;
  const long long span = (hw + chunks - 1) / chunks;
  chunks = (hw + span - 1) / span;
  return {dim3(static_cast<unsigned>(chunks), static_cast<unsigned>(n)), dim3(bx, by), span};
}

bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

bool slope_act(int a) { return a == GAP_ACT_NONE || a == GAP_ACT_LRELU || a == GAP_ACT_RELU; }

// the shape checks every entry point shares; sets the error message and returns false on a bad shape
bool in_shape_ok(const char* fn, int n, int64_t hw, int c, int64_t ld) {
  if (n < 1 || n > 65535 || hw < 2 || c < 8 || c > kInMaxC || c % 8 != 0 || ld < c || ld % 8 != 0) {
    set_error("%s: bad arguments (need 1 <= n <= 65535, H*W >= 2, C %% 8 == 0 with 8 <= C <= %d, pixel stride >= C "
              "and a multiple of 8; got n=%d hw=%lld c=%d ld=%lld)", fn, kInMaxC, n, static_cast<long long>(hw), c,
              static_cast<long long>(ld));
    return false;
  }
  return true;
}

int in_bwd_launch(bool apply, InBwdArgs a, int n, cudaStream_t st) {
  const InGeom g = in_geom(n, a.hw, a.c);
  a.span = g.span;
  const size_t smem = apply ? (a.dbias ? static_cast<size_t>(g.block.y) * a.c * sizeof(float) : 0)
                            : static_cast<size_t>(g.block.y) * a.c * 2 * sizeof(float);
  const bool g2 = a.g2 != nullptr;
  if (apply) {
    if (g2)
      GAP_CUDA(launch_pdl(in_bwd_kernel<true, true>, g.grid, g.block, smem, st, a));
    else
      GAP_CUDA(launch_pdl(in_bwd_kernel<true, false>, g.grid, g.block, smem, st, a));
  } else {
    if (g2)
      GAP_CUDA(launch_pdl(in_bwd_kernel<false, true>, g.grid, g.block, smem, st, a));
    else
      GAP_CUDA(launch_pdl(in_bwd_kernel<false, false>, g.grid, g.block, smem, st, a));
  }
  GAP_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace
}  // namespace gap

using namespace gap;

extern "C" {

int gap_in_stats(const void* y, int64_t ld, int n, int64_t hw, int c, double* sums, void* stream) {
  GAP_CHECK_ARG(y && sums, "gap_in_stats: null pointer");
  if (!in_shape_ok("gap_in_stats", n, hw, c, ld)) return GAP_ERR_BAD_ARG;
  GAP_CHECK_ARG(al16(y), "gap_in_stats: y must be 16-byte aligned");
  const InGeom g = in_geom(n, hw, c);
  const size_t smem = static_cast<size_t>(g.block.y) * c * 2 * sizeof(float);
  GAP_CUDA(launch_pdl(in_stats_kernel, g.grid, g.block, smem, static_cast<cudaStream_t>(stream),
                      static_cast<const bf16*>(y), static_cast<long long>(ld), static_cast<long long>(hw), c, g.span, sums,
                      n * c));
  GAP_CUDA(cudaGetLastError());
  return 0;
}

int gap_in_act(const void* y, int64_t ld, int n, int64_t hw, int c, const float* scale, const float* shift, void* out1,
               int64_t ld1, int act1, void* out2, int64_t ld2, int act2, void* stream) {
  GAP_CHECK_ARG(y && scale && shift && out1, "gap_in_act: null pointer");
  if (!in_shape_ok("gap_in_act", n, hw, c, ld)) return GAP_ERR_BAD_ARG;
  GAP_CHECK_ARG(slope_act(act1) && (!out2 || slope_act(act2)), "gap_in_act: act must be NONE, LRELU or RELU");
  GAP_CHECK_ARG(ld1 >= c && ld1 % 8 == 0 && (!out2 || (ld2 >= c && ld2 % 8 == 0)),
                "gap_in_act: output pixel strides must be >= C and multiples of 8");
  GAP_CHECK_ARG(al16(y) && al16(out1) && al16(out2), "gap_in_act: tensors must be 16-byte aligned");
  const InGeom g = in_geom(n, hw, c);
  GAP_CUDA(launch_pdl(in_act_kernel, g.grid, g.block, 0, static_cast<cudaStream_t>(stream), static_cast<const bf16*>(y),
                      static_cast<long long>(ld), static_cast<long long>(hw), c, g.span, scale, shift,
                      static_cast<bf16*>(out1), static_cast<long long>(ld1), act1, static_cast<bf16*>(out2),
                      static_cast<long long>(ld2), act2));
  GAP_CUDA(cudaGetLastError());
  return 0;
}

int gap_in_bwd_reduce(const void* y, int64_t ld, const void* g1, int64_t ld_g1, const void* g2, int64_t ld_g2, float slope,
                      const float* scale, const float* shift, int n, int64_t hw, int c, double* sums, void* stream) {
  GAP_CHECK_ARG(y && g1 && scale && shift && sums, "gap_in_bwd_reduce: null pointer");
  if (!in_shape_ok("gap_in_bwd_reduce", n, hw, c, ld)) return GAP_ERR_BAD_ARG;
  GAP_CHECK_ARG(ld_g1 >= c && ld_g1 % 8 == 0 && (!g2 || (ld_g2 >= c && ld_g2 % 8 == 0)),
                "gap_in_bwd_reduce: gradient pixel strides must be >= C and multiples of 8");
  GAP_CHECK_ARG(al16(y) && al16(g1) && al16(g2), "gap_in_bwd_reduce: tensors must be 16-byte aligned");
  const InBwdArgs a{static_cast<const bf16*>(y), ld, static_cast<const bf16*>(g1), ld_g1, static_cast<const bf16*>(g2),
                    ld_g2, slope, scale, shift, hw, c, n * c, 0, sums, 0.0, nullptr, 0, nullptr};
  return in_bwd_launch(false, a, n, static_cast<cudaStream_t>(stream));
}

int gap_in_bwd_apply(const void* y, int64_t ld, const void* g1, int64_t ld_g1, const void* g2, int64_t ld_g2, float slope,
                     const float* scale, const float* shift, int n, int64_t hw, int c, const double* sums, void* dy,
                     int64_t ld_dy, float* dbias, void* stream) {
  GAP_CHECK_ARG(y && g1 && scale && shift && sums && dy, "gap_in_bwd_apply: null pointer");
  if (!in_shape_ok("gap_in_bwd_apply", n, hw, c, ld)) return GAP_ERR_BAD_ARG;
  GAP_CHECK_ARG(ld_g1 >= c && ld_g1 % 8 == 0 && (!g2 || (ld_g2 >= c && ld_g2 % 8 == 0)) && ld_dy >= c && ld_dy % 8 == 0,
                "gap_in_bwd_apply: pixel strides must be >= C and multiples of 8");
  GAP_CHECK_ARG(al16(y) && al16(g1) && al16(g2) && al16(dy), "gap_in_bwd_apply: tensors must be 16-byte aligned");
  const InBwdArgs a{static_cast<const bf16*>(y), ld, static_cast<const bf16*>(g1), ld_g1, static_cast<const bf16*>(g2),
                    ld_g2, slope, scale, shift, hw, c, n * c, 0, const_cast<double*>(sums), 1.0 / static_cast<double>(hw),
                    static_cast<bf16*>(dy), ld_dy, dbias};
  return in_bwd_launch(true, a, n, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
