// Sliding-window inference of the Siamese U-Net over a whole scene (SiameseEngine.predict_scene): the scene is cut into
// overlapping tiles of one fixed extent, the tiles run in batches through the eval-mode network, and their class
// probabilities are blended with a Gaussian window into full-resolution accumulators.
//
// Tile grid, per axis (scene length L, tile T, overlap o; siamese.scene_axis is the same definition in Python):
//   L <= T: one tile at origin 0 with extent E = ceil16(L); reads past L clamp to the last row / column.
//   L >  T: E = T, step S = T - o, n = ceil((L - T) / S) + 1 tiles at origins min(i S, L - T).
// Tiles are numbered row-major over the grid.  The kernels take the per-axis (L, E, S, n) and derive every origin from
// the tile index, so no per-batch table travels from the host.
// Window: w(ty, tx) = g_y(ty) g_x(tx), g(t) = exp(-(t + 0.5 - E/2)^2 / (2 sigma^2)), sigma = E/8.
//
// gap_scene_gather   scene pixels (uint8 HWC or fp32 CHW) -> the engine's two 4-slot NHWC bf16 input batches
// gap_scene_blend    logits of one batch -> acc[K][H][W] += w p, wsum[H][W] += w (gather form, no float atomics)
// gap_scene_finalize acc / wsum -> uint8 pred (argmax or > 0.5), optional in-place probabilities, confusion counts
#include <algorithm>

#include "common.h"
#include "ptx.cuh"

namespace gap {

typedef __nv_bfloat16 bf16;

constexpr int kSceneMaxClasses = 16;

struct SceneAxis {
  int len, ext, step, n;
};

__device__ __forceinline__ int axis_origin(const SceneAxis& a, int i) {
  return a.n == 1 ? 0 : min(i * a.step, a.len - a.ext);
}

// The tiles [first, last] of one axis that cover scene coordinate v (0 <= v < len).  Origins never decrease and every
// extent is the same, so the covering tiles are contiguous; tile i < n-1 sits at i*step, the last one at len - ext.
__device__ __forceinline__ void axis_cover(const SceneAxis& a, int v, int& first, int& last) {
  int lo = v >= a.ext ? (v - a.ext) / a.step + 1 : 0;
  lo = min(lo, a.n - 1);
  int hi = lo;
  while (hi + 1 < a.n && axis_origin(a, hi + 1) <= v) ++hi;
  first = lo;
  last = hi;
}

// g(t) of an axis of extent e: exp(-(t + 0.5 - e/2)^2 / (2 (e/8)^2)) = exp(-32 d^2 / e^2)
__device__ __forceinline__ float window(int t, int e) {
  const float d = t + 0.5f - 0.5f * e;
  return expf(-32.f * d * d / (static_cast<float>(e) * e));
}

// ------------------------------------------------------------------------------------------------
// Gather: one thread per pixel of the batch, both scenes.  Tile index tile0 + b >= ny*nx is a padding tile (zeros).
// The values are those of gap_u8_hwc_to_nhwc_bf16_c (x * 2/255 - 1) / gap_nchw_f32_to_nhwc_bf16 (round to nearest) on
// the same crop; slots >= C are zero.
// ------------------------------------------------------------------------------------------------
template <int C, bool U8>
__global__ void __launch_bounds__(256) scene_gather_kernel(const void* __restrict__ img1, const void* __restrict__ img2,
                                                           SceneAxis ay, SceneAxis ax, int tile0, int batch,
                                                           bf16* __restrict__ out1, bf16* __restrict__ out2) {
  const long long per_tile = static_cast<long long>(ay.ext) * ax.ext;
  const long long total = per_tile * batch;
  const long long hw = static_cast<long long>(ay.len) * ax.len;
  const int n_tiles = ay.n * ax.n;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int b = static_cast<int>(i / per_tile);
    const int r = static_cast<int>(i - b * per_tile);
    const int t = tile0 + b;
    float v1[4] = {0.f, 0.f, 0.f, 0.f}, v2[4] = {0.f, 0.f, 0.f, 0.f};
    if (t < n_tiles) {
      const int ty = t / ax.n, tx = t - ty * ax.n;
      const int y = min(axis_origin(ay, ty) + r / ax.ext, ay.len - 1);
      const int x = min(axis_origin(ax, tx) + r % ax.ext, ax.len - 1);
      const long long p = static_cast<long long>(y) * ax.len + x;
      if (U8) {
        const uint8_t* s1 = static_cast<const uint8_t*>(img1) + p * C;
        const uint8_t* s2 = static_cast<const uint8_t*>(img2) + p * C;
#pragma unroll
        for (int j = 0; j < C; ++j) {
          v1[j] = s1[j] * (2.f / 255.f) - 1.f;
          v2[j] = s2[j] * (2.f / 255.f) - 1.f;
        }
      } else {
        const float* s1 = static_cast<const float*>(img1) + p;
        const float* s2 = static_cast<const float*>(img2) + p;
#pragma unroll
        for (int j = 0; j < C; ++j) {
          v1[j] = __ldg(s1 + j * hw);
          v2[j] = __ldg(s2 + j * hw);
        }
      }
    }
    *reinterpret_cast<uint2*>(out1 + i * 4) = make_uint2(pack_bf16x2(v1[0], v1[1]), pack_bf16x2(v1[2], v1[3]));
    *reinterpret_cast<uint2*>(out2 + i * 4) = make_uint2(pack_bf16x2(v2[0], v2[1]), pack_bf16x2(v2[2], v2[3]));
  }
}

// ------------------------------------------------------------------------------------------------
// Blend, gather form: one thread per scene pixel of the box [y0, y0+bh) x [x0, x0+bw) that the batch's tiles
// [t0, t1) cover.  The thread visits the tiles of the batch that cover its pixel in ascending index and adds w*p and w
// onto the running sums, one fused multiply-add per tile, so each pixel sees the same sequence of operations whatever
// the batch size.  When the first tile of the whole grid that covers the pixel is in this batch the sums start from
// zero (the accumulators need no clearing), otherwise from what the earlier batches stored.  KT: the class count when
// fixed at compile time (1 = sigmoid), 0 = runtime k <= 16.
// ------------------------------------------------------------------------------------------------
template <int KT>
__global__ void __launch_bounds__(256) scene_blend_kernel(const float* __restrict__ logits, int k, SceneAxis ay,
                                                          SceneAxis ax, int t0, int t1, int y0, int x0, int bh, int bw,
                                                          float* __restrict__ acc, float* __restrict__ wsum) {
  constexpr int KM = KT > 0 ? KT : kSceneMaxClasses;
  const int K = KT > 0 ? KT : k;
  const long long total = static_cast<long long>(bh) * bw;
  const long long hw = static_cast<long long>(ay.len) * ax.len;
  const long long tile_px = static_cast<long long>(ay.ext) * ax.ext;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int Y = y0 + static_cast<int>(i / bw), X = x0 + static_cast<int>(i % bw);
    int ya, yb, xa, xb;
    axis_cover(ay, Y, ya, yb);
    axis_cover(ax, X, xa, xb);
    if ((yb * ax.n + xb) < t0 || (ya * ax.n + xa) >= t1) continue;
    const long long p = static_cast<long long>(Y) * ax.len + X;
    float a[KM];
    float ws = 0.f;
    const bool fresh = ya * ax.n + xa >= t0;
#pragma unroll
    for (int c = 0; c < KM; ++c) a[c] = (c < K && !fresh) ? acc[c * hw + p] : 0.f;
    if (!fresh) ws = wsum[p];
    bool any = false;
    for (int ty = ya; ty <= yb; ++ty) {
      const int oy = axis_origin(ay, ty);
      const float gy = window(Y - oy, ay.ext);
      for (int tx = xa; tx <= xb; ++tx) {
        const int t = ty * ax.n + tx;
        if (t < t0 || t >= t1) continue;
        any = true;
        const int ox = axis_origin(ax, tx);
        const float w = gy * window(X - ox, ax.ext);
        const float* lg = logits + (t - t0) * K * tile_px + static_cast<long long>(Y - oy) * ax.ext + (X - ox);
        if (KT == 1) {
          const float pr = 1.f / (1.f + expf(-__ldg(lg)));
          a[0] = fmaf(w, pr, a[0]);
        } else {
          float v[KM];
          float m = -INFINITY;
#pragma unroll
          for (int c = 0; c < KM; ++c)
            if (c < K) {
              v[c] = __ldg(lg + c * tile_px);
              m = fmaxf(m, v[c]);
            }
          float se = 0.f;
#pragma unroll
          for (int c = 0; c < KM; ++c)
            if (c < K) {
              v[c] = expf(v[c] - m);
              se += v[c];
            }
          const float inv = 1.f / se;
#pragma unroll
          for (int c = 0; c < KM; ++c)
            if (c < K) a[c] = fmaf(w, v[c] * inv, a[c]);
        }
        ws += w;
      }
    }
    if (!any) continue;
#pragma unroll
    for (int c = 0; c < KM; ++c)
      if (c < K) acc[c * hw + p] = a[c];
    wsum[p] = ws;
  }
}

// ------------------------------------------------------------------------------------------------
// Finalize: p = acc / wsum; pred = argmax_c p (ties to the lowest class, NaN above everything, as torch.argmax) or
// p > 0.5 for K = 1; probs (optional) overwrite acc in place.  Confusion counts (labels given): K > 1 counts[label][pred],
// K = 1 counts[TP, FP, FN, TN] with label 1 positive and 0 negative; ignore_index and labels outside the class range
// are skipped.  Shared-memory histogram per CTA (equal bins of a warp added once), one 64-bit atomic per bin and CTA.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool scene_better(float v, float bv) {
  const bool vn = v != v, bn = bv != bv;
  if (vn != bn) return vn;
  return !vn && v > bv;
}

template <int KT>
__global__ void __launch_bounds__(256) scene_finalize_kernel(float* __restrict__ acc, const float* __restrict__ wsum,
                                                             int k, long long hw, uint8_t* __restrict__ pred,
                                                             int write_probs, const long long* __restrict__ labels,
                                                             long long ignore, unsigned long long* __restrict__ counts) {
  constexpr int KM = KT > 0 ? KT : kSceneMaxClasses;
  const int K = KT > 0 ? KT : k;
  const int bins = K == 1 ? 4 : K * K;
  __shared__ unsigned int hist[kSceneMaxClasses * kSceneMaxClasses];
  if (labels) {
    for (int i = threadIdx.x; i < bins; i += blockDim.x) hist[i] = 0u;
    __syncthreads();
  }
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i0 = blockIdx.x * static_cast<long long>(blockDim.x); i0 < hw; i0 += stride) {   // uniform per warp
    const long long i = i0 + threadIdx.x;
    int bin = -1;
    if (i < hw) {
      const float inv = 1.f / wsum[i];
      int best = 0;
      if (KT == 1) {
        const float pr = acc[i] * inv;
        best = pr > 0.5f ? 1 : 0;
        if (write_probs) acc[i] = pr;
      } else {
        float bv = 0.f;
#pragma unroll
        for (int c = 0; c < KM; ++c)
          if (c < K) {
            const float pr = acc[c * hw + i] * inv;
            if (c == 0 || scene_better(pr, bv)) {
              bv = pr;
              best = c;
            }
            if (write_probs) acc[c * hw + i] = pr;
          }
      }
      pred[i] = static_cast<uint8_t>(best);
      if (labels) {
        const long long y = labels[i];
        if (y != ignore && y >= 0 && y < (K == 1 ? 2 : K))
          bin = K == 1 ? (y == 1 ? (best ? 0 : 2) : (best ? 1 : 3)) : static_cast<int>(y) * K + best;
      }
    }
    if (labels) {
      const unsigned int peers = __match_any_sync(0xffffffffu, bin);
      if (bin >= 0 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&hist[bin], __popc(peers));
    }
  }
  if (labels) {
    __syncthreads();
    for (int i = threadIdx.x; i < bins; i += blockDim.x)
      if (hist[i]) atomicAdd(counts + i, static_cast<unsigned long long>(hist[i]));
  }
}

static inline int scene_grid(long long work, int max_blocks) {
  long long g = (work + 255) / 256;
  if (g < 1) g = 1;
  return static_cast<int>(std::min<long long>(g, max_blocks));
}

static inline bool scene_axis_ok(const SceneAxis& a) {
  return a.len >= 1 && a.ext >= 16 && a.ext % 16 == 0 && a.n >= 1 && a.step >= 1 && a.step <= a.ext &&
         (a.n == 1 ? a.len <= a.ext : a.len > a.ext && static_cast<long long>(a.n - 1) * a.step >= a.len - a.ext &&
                                          static_cast<long long>(a.n - 2) * a.step < a.len - a.ext);
}

static inline int scene_origin_host(const SceneAxis& a, int i) { return a.n == 1 ? 0 : std::min(i * a.step, a.len - a.ext); }

}  // namespace gap

using namespace gap;

extern "C" {

int gap_scene_gather(const void* img1, const void* img2, int src_u8, int c, int h, int w, int ey, int ex, int sy,
                     int sx, int ny, int nx, int tile0, int batch, void* out1, void* out2, void* stream) {
  GAP_CHECK_ARG(c >= 1 && c <= 4, "gap_scene_gather: c must be 1..4, got %d", c);
  const SceneAxis ay{h, ey, sy, ny}, ax{w, ex, sx, nx};
  GAP_CHECK_ARG(img1 && img2 && out1 && out2 && scene_axis_ok(ay) && scene_axis_ok(ax) && batch >= 1 && tile0 >= 0 &&
                    tile0 < ny * nx,
                "gap_scene_gather: bad arguments");
  GAP_CHECK_ARG((reinterpret_cast<uintptr_t>(out1) & 7) == 0 && (reinterpret_cast<uintptr_t>(out2) & 7) == 0,
                "gap_scene_gather: out1 / out2 must be 8-byte aligned (one 8-byte store per 4-slot pixel)");
  const long long total = static_cast<long long>(ey) * ex * batch;
  const int grid = scene_grid(total, 148 * 8);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  bf16* o1 = static_cast<bf16*>(out1);
  bf16* o2 = static_cast<bf16*>(out2);
#define GATHER(CC, U)                                                                                     \
  scene_gather_kernel<CC, U><<<grid, 256, 0, st>>>(img1, img2, ay, ax, tile0, batch, o1, o2)
  if (src_u8) {
    switch (c) {
      case 1: GATHER(1, true); break;
      case 2: GATHER(2, true); break;
      case 3: GATHER(3, true); break;
      default: GATHER(4, true); break;
    }
  } else {
    switch (c) {
      case 1: GATHER(1, false); break;
      case 2: GATHER(2, false); break;
      case 3: GATHER(3, false); break;
      default: GATHER(4, false); break;
    }
  }
#undef GATHER
  GAP_CUDA(cudaGetLastError());
  return 0;
}

int gap_scene_blend(const float* logits, int k, int h, int w, int ey, int ex, int sy, int sx, int ny, int nx, int tile0,
                    int batch, float* acc, float* wsum, void* stream) {
  GAP_CHECK_ARG(k >= 1 && k <= kSceneMaxClasses, "gap_scene_blend: k must be 1..16, got %d", k);
  const SceneAxis ay{h, ey, sy, ny}, ax{w, ex, sx, nx};
  GAP_CHECK_ARG(logits && acc && wsum && scene_axis_ok(ay) && scene_axis_ok(ax) && batch >= 1 && tile0 >= 0 &&
                    tile0 < ny * nx,
                "gap_scene_blend: bad arguments");
  const int t0 = tile0, t1 = std::min(tile0 + batch, ny * nx);
  // the box the batch's tiles cover: their tile rows, and their columns when they share one tile row
  const int ty0 = t0 / nx, ty1 = (t1 - 1) / nx;
  const int y0 = scene_origin_host(ay, ty0), y1 = std::min(scene_origin_host(ay, ty1) + ey, h);
  int x0 = 0, x1 = w;
  if (ty0 == ty1) {
    x0 = scene_origin_host(ax, t0 - ty0 * nx);
    x1 = std::min(scene_origin_host(ax, t1 - 1 - ty0 * nx) + ex, w);
  }
  const int bh = y1 - y0, bw = x1 - x0;
  const int grid = scene_grid(static_cast<long long>(bh) * bw, 148 * 8);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (k) {
    case 1: scene_blend_kernel<1><<<grid, 256, 0, st>>>(logits, k, ay, ax, t0, t1, y0, x0, bh, bw, acc, wsum); break;
    case 2: scene_blend_kernel<2><<<grid, 256, 0, st>>>(logits, k, ay, ax, t0, t1, y0, x0, bh, bw, acc, wsum); break;
    default: scene_blend_kernel<0><<<grid, 256, 0, st>>>(logits, k, ay, ax, t0, t1, y0, x0, bh, bw, acc, wsum); break;
  }
  GAP_CUDA(cudaGetLastError());
  return 0;
}

int gap_scene_finalize(float* acc, const float* wsum, int k, int64_t pixels, uint8_t* pred, int write_probs,
                       const int64_t* labels, int64_t ignore_index, int64_t* counts, void* stream) {
  GAP_CHECK_ARG(k >= 1 && k <= kSceneMaxClasses, "gap_scene_finalize: k must be 1..16, got %d", k);
  GAP_CHECK_ARG(acc && wsum && pred && pixels > 0 && (labels == nullptr) == (counts == nullptr),
                "gap_scene_finalize: bad arguments");
  const int grid = scene_grid(pixels, 148 * 8);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long* lab = reinterpret_cast<const long long*>(labels);
  unsigned long long* cnt = reinterpret_cast<unsigned long long*>(counts);
  switch (k) {
    case 1: scene_finalize_kernel<1><<<grid, 256, 0, st>>>(acc, wsum, k, pixels, pred, write_probs, lab, ignore_index, cnt); break;
    case 2: scene_finalize_kernel<2><<<grid, 256, 0, st>>>(acc, wsum, k, pixels, pred, write_probs, lab, ignore_index, cnt); break;
    default: scene_finalize_kernel<0><<<grid, 256, 0, st>>>(acc, wsum, k, pixels, pred, write_probs, lab, ignore_index, cnt); break;
  }
  GAP_CUDA(cudaGetLastError());
  return 0;
}

}  // extern "C"
