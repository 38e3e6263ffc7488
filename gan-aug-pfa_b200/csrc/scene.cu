// Sliding-window inference over a whole scene: the scene is cut into overlapping tiles of one fixed extent, the tiles
// run in batches through an eval-mode network, and its per-tile outputs are blended with a Gaussian window into
// full-resolution accumulators.  Two networks use it: the Siamese U-Net (SiameseEngine.predict_scene: class
// probabilities of an image pair) and the Pix2Pix generator (GeneratorEngine.translate_scene: the Tanh image).
//
// Tile grid, per axis (scene length L, tile T, overlap o, alignment A; scene.scene_axis is the same definition in
// Python, A = 16 for the Siamese U-Net and 2^depth for the generator):
//   L <= T: one tile at origin 0 with extent E = L rounded up to A; reads past L clamp to the last row / column.
//   L >  T: E = T, step S = T - o, n = ceil((L - T) / S) + 1 tiles at origins min(i S, L - T).
// Tiles are numbered row-major over the grid.  The kernels take the per-axis (L, E, S, n) and derive every origin from
// the tile index, so no per-batch table travels from the host.
// Window: w(ty, tx) = g_y(ty) g_x(tx), g(t) = exp(-(t + 0.5 - E/2)^2 / (2 sigma^2)), sigma = E/8.
//
// gap_scene_gather   scene pixels (uint8 HWC or fp32 CHW) -> the engine's two 4-slot NHWC bf16 input batches
// gap_scene_blend    logits of one batch -> acc[K][H][W] += w p, wsum[H][W] += w (gather form, no float atomics)
// gap_scene_finalize acc / wsum -> uint8 pred (argmax or > 0.5), optional in-place probabilities, confusion counts
// gap_scene_gather_tta / gap_scene_blend_tta  the same gather and blend for a dihedral transform d of every tile, and
//                    a blend that keeps adding over several passes (test-time augmentation, checkpoint ensembles)
// gap_scene_gather_one      one scene -> the generator's 4-slot NHWC bf16 input batch
// gap_scene_blend_image     generator output of one batch (fp32 [batch][ey][ex][4]) -> acc[C][H][W] += w v, wsum += w
// gap_scene_finalize_image  acc / wsum -> uint8 image [H][W][C] (the Tanh output's 8-bit rule), optional in-place values
#include <algorithm>

#include "common.h"
#include "confusion.cuh"
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

// The tiles of one batch [t0, t1) that cover scene pixel (Y, X): the covering range of each axis, and `fresh` when the
// pixel's first covering tile of the whole grid is in the batch (its sums then start from zero, so the accumulators
// need no clearing).  False when every covering tile lies before t0 or from t1 on.
struct PixelCover {
  int ya, yb, xa, xb;
  bool fresh;
};

__device__ __forceinline__ bool batch_cover(const SceneAxis& ay, const SceneAxis& ax, int Y, int X, int t0, int t1,
                                            PixelCover& c) {
  axis_cover(ay, Y, c.ya, c.yb);
  axis_cover(ax, X, c.xa, c.xb);
  if (c.yb * ax.n + c.xb < t0 || c.ya * ax.n + c.xa >= t1) return false;
  c.fresh = c.ya * ax.n + c.xa >= t0;
  return true;
}

// Visits the tiles of the batch that cover (Y, X) in ascending index: f(b, ty, tx, w) with b = t - t0 the tile's slot
// in the batch, (ty, tx) the pixel inside the tile and w = gy(ty) * gx(tx) its window weight (gy, gx: the per-axis
// window, evaluated or looked up).  Returns whether any tile was visited.
template <class GY, class GX, class F>
__device__ __forceinline__ bool visit_batch_tiles(const SceneAxis& ay, const SceneAxis& ax, int Y, int X, int t0,
                                                  int t1, const PixelCover& c, GY gy, GX gx, F f) {
  bool any = false;
  for (int ty = c.ya; ty <= c.yb; ++ty) {
    const int row = ty * ax.n;                     // the covering tiles of this tile row that are in [t0, t1)
    const int xa = max(c.xa, t0 - row), xb = min(c.xb, t1 - 1 - row);
    if (xa > xb) continue;
    any = true;
    const int oy = axis_origin(ay, ty);
    const float wy = gy(Y - oy);
    for (int tx = xa; tx <= xb; ++tx) {
      const int ox = axis_origin(ax, tx);
      f(row + tx - t0, Y - oy, X - ox, wy * gx(X - ox));
    }
  }
  return any;
}

// ------------------------------------------------------------------------------------------------
// Dihedral tile transforms (test-time augmentation).  d = 4 s + 2 v + u: f_d transposes the tile's two axes if s, then
// flips its rows if v, then its columns if u, so the network sees [ex][ey] when s = 1.  Pixel (ty, tx) of a tile sits
// at (i, j) of f_d(tile) with (i, j) = (s ? tx : ty, s ? ty : tx), i -> OY-1-i if v, j -> OX-1-j if u, where
// [OY][OX] is the transformed extent; the logits of f_d(tile) are read back at the same (i, j) (the map f_d^-1).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ long long tta_offset(int d, int ty, int tx, int ey, int ex) {
  const bool s = d & 4;
  const int oy = s ? ex : ey, ox = s ? ey : ex;
  int i = s ? tx : ty, j = s ? ty : tx;
  if (d & 2) i = oy - 1 - i;
  if (d & 1) j = ox - 1 - j;
  return static_cast<long long>(i) * ox + j;
}

// The 4-slot values of scene pixel p: gap_u8_hwc_to_nhwc_bf16_c (x * 2/255 - 1) or gap_nchw_f32_to_nhwc_bf16 (round to
// nearest) of the same pixel, slots >= C zero, packed as one 8-byte NHWC bf16 pixel.
template <int C, bool U8>
__device__ __forceinline__ uint2 scene_pixel(const void* img, long long p, long long hw) {
  float v[4] = {0.f, 0.f, 0.f, 0.f};
  if (U8) {
    const uint8_t* s = static_cast<const uint8_t*>(img) + p * C;
#pragma unroll
    for (int j = 0; j < C; ++j) v[j] = s[j] * (2.f / 255.f) - 1.f;
  } else {
    const float* s = static_cast<const float*>(img) + p;
#pragma unroll
    for (int j = 0; j < C; ++j) v[j] = __ldg(s + j * hw);
  }
  return make_uint2(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]));
}

// ------------------------------------------------------------------------------------------------
// Gather, NIMG = 1 or 2 scenes, of f_d of every tile (d < 4 when S = false, d >= 4 when S = true).  Tile index
// tile0 + b >= ny*nx is a padding tile (zeros).
// S = false: one thread per output pixel; consecutive threads read consecutive (or, flipped, reversed) scene columns.
// S = true (transposed tiles): one CTA of 256 threads per 16 x 16 square of an output tile.  The threads first read
// the square's source pixels along scene rows into shared memory, then write the output square row by row from there,
// so both the scene reads and the output writes stay coalesced.  Extents are multiples of 16: squares are whole.
// ------------------------------------------------------------------------------------------------
template <int C, bool U8, int NIMG, bool S>
__global__ void __launch_bounds__(256) scene_gather_kernel(const void* __restrict__ img1, const void* __restrict__ img2,
                                                           SceneAxis ay, SceneAxis ax, int tile0, int batch, int d,
                                                           bf16* __restrict__ out1, bf16* __restrict__ out2) {
  const long long per_tile = static_cast<long long>(ay.ext) * ax.ext;
  const long long hw = static_cast<long long>(ay.len) * ax.len;
  const int n_tiles = ay.n * ax.n;
  const void* img[2] = {img1, img2};
  bf16* out[2] = {out1, out2};
  const int oy = S ? ax.ext : ay.ext, ox = S ? ay.ext : ax.ext;       // the transformed extent [oy][ox]
  if constexpr (!S) {
    const long long total = per_tile * batch;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
      const int b = static_cast<int>(i / per_tile);
      const int r = static_cast<int>(i - b * per_tile);
      const int t = tile0 + b;
      uint2 v[NIMG];
#pragma unroll
      for (int m = 0; m < NIMG; ++m) v[m] = make_uint2(0u, 0u);
      if (t < n_tiles) {
        const int ty = t / ax.n, tx = t - ty * ax.n;
        const int ri = r / ox, rj = r % ox;
        const int y = min(axis_origin(ay, ty) + ((d & 2) ? oy - 1 - ri : ri), ay.len - 1);
        const int x = min(axis_origin(ax, tx) + ((d & 1) ? ox - 1 - rj : rj), ax.len - 1);
        const long long p = static_cast<long long>(y) * ax.len + x;
#pragma unroll
        for (int m = 0; m < NIMG; ++m) v[m] = scene_pixel<C, U8>(img[m], p, hw);
      }
#pragma unroll
      for (int m = 0; m < NIMG; ++m) *reinterpret_cast<uint2*>(out[m] + i * 4) = v[m];
    }
  } else {
    __shared__ uint2 sq[NIMG][16][17];                  // [source row][source column] of one square, padded
    const int sqx = ox / 16, per_tile_sq = (oy / 16) * sqx;
    const int lo = threadIdx.x & 15, hi = threadIdx.x >> 4;
    for (int q = blockIdx.x; q < batch * per_tile_sq; q += gridDim.x) {   // uniform per CTA
      const int b = q / per_tile_sq, qs = q - b * per_tile_sq;
      const int r0 = (qs / sqx) * 16, c0 = (qs % sqx) * 16;        // the output square [r0, r0+16) x [c0, c0+16)
      const int t = tile0 + b;
      // its source: tile rows ty = c0.. (or, flipped, ox-16-c0..), tile columns tx = r0.. (or oy-16-r0..)
      const int sy0 = (d & 1) ? ox - 16 - c0 : c0, sx0 = (d & 2) ? oy - 16 - r0 : r0;
      const bool real = t < n_tiles;
      __syncthreads();                                 // the previous square's reads of sq are done
      if (real) {
        const int ty = t / ax.n, tx = t - ty * ax.n;
        const int y = min(axis_origin(ay, ty) + sy0 + hi, ay.len - 1);
        const int x = min(axis_origin(ax, tx) + sx0 + lo, ax.len - 1);
        const long long p = static_cast<long long>(y) * ax.len + x;
#pragma unroll
        for (int m = 0; m < NIMG; ++m) sq[m][hi][lo] = scene_pixel<C, U8>(img[m], p, hw);
      }
      __syncthreads();
      // output pixel (r0 + hi, c0 + lo) is tile pixel (ty, tx) = (c', r') with c' = c0 + lo or ox-1-(c0 + lo) and
      // r' = r0 + hi or oy-1-(r0 + hi); relative to the source square that is (lo or 15 - lo, hi or 15 - hi)
      const int a = (d & 1) ? 15 - lo : lo, bb = (d & 2) ? 15 - hi : hi;
      const long long o = (static_cast<long long>(b) * per_tile + static_cast<long long>(r0 + hi) * ox + c0 + lo) * 4;
#pragma unroll
      for (int m = 0; m < NIMG; ++m)
        *reinterpret_cast<uint2*>(out[m] + o) = real ? sq[m][a][bb] : make_uint2(0u, 0u);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Blend, gather form, over the scene pixels of the box [y0, y0+bh) x [x0, x0+bw) that the batch's tiles [t0, t1)
// cover.  Each pixel visits the tiles of the batch that cover it in ascending index and adds w*p and w onto its
// running sums, one fused multiply-add per tile, so each pixel sees the same sequence of operations whatever the batch
// size.  When the first tile of the whole grid that covers the pixel is in this batch and this is the first pass the
// sums start from zero (the accumulators need no clearing), otherwise from what the earlier batches and passes stored.
// The logits are those of f_d(tile) (tta_offset).  KT: the class count when fixed at compile time (1 = sigmoid),
// 0 = runtime k <= 16.
// S = false (d < 4): one thread per pixel, consecutive threads on consecutive (flipped: reversed) tile columns.
// S = true (d >= 4, logits [ex][ey] per class plane): one CTA per 16 x 16 box of pixels.  For each batch tile that
// covers part of the box, in ascending index, the threads first copy the box's logits into shared memory with
// consecutive threads on consecutive scene rows (consecutive addresses of the transposed plane), then every thread
// reads its pixel's K values from there; the per-pixel arithmetic is that of S = false.
// ------------------------------------------------------------------------------------------------
template <int KT, class LD>
__device__ __forceinline__ void blend_tile(LD ld, int K, float w, float* a) {
  constexpr int KM = KT > 0 ? KT : kSceneMaxClasses;
  if (KT == 1) {
    const float pr = 1.f / (1.f + expf(-ld(0)));
    a[0] = fmaf(w, pr, a[0]);
  } else {
    float v[KM];
    float m = -INFINITY;
#pragma unroll
    for (int c = 0; c < KM; ++c)
      if (c < K) {
        v[c] = ld(c);
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
}

template <int KT, bool S>
__global__ void __launch_bounds__(256) scene_blend_kernel(const float* __restrict__ logits, int k, SceneAxis ay,
                                                          SceneAxis ax, int t0, int t1, int y0, int x0, int bh, int bw,
                                                          int d, int first_pass, float* __restrict__ acc,
                                                          float* __restrict__ wsum) {
  constexpr int KM = KT > 0 ? KT : kSceneMaxClasses;
  const int K = KT > 0 ? KT : k;
  const long long hw = static_cast<long long>(ay.len) * ax.len;
  const long long tile_px = static_cast<long long>(ay.ext) * ax.ext;
  auto gy = [&](int t) { return window(t, ay.ext); };
  auto gx = [&](int t) { return window(t, ax.ext); };
  if constexpr (!S) {
    const long long total = static_cast<long long>(bh) * bw;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
      const int Y = y0 + static_cast<int>(i / bw), X = x0 + static_cast<int>(i % bw);
      PixelCover cv;
      if (!batch_cover(ay, ax, Y, X, t0, t1, cv)) continue;
      const bool fresh = cv.fresh && first_pass;
      const long long p = static_cast<long long>(Y) * ax.len + X;
      float a[KM];
      float ws = 0.f;
#pragma unroll
      for (int c = 0; c < KM; ++c) a[c] = (c < K && !fresh) ? acc[c * hw + p] : 0.f;
      if (!fresh) ws = wsum[p];
      const bool any = visit_batch_tiles(ay, ax, Y, X, t0, t1, cv, gy, gx, [&](int b, int ty, int tx, float w) {
        const float* lg = logits + b * K * tile_px + tta_offset(d, ty, tx, ay.ext, ax.ext);
        blend_tile<KT>([&](int c) { return __ldg(lg + c * tile_px); }, K, w, a);
        ws += w;
      });
      if (!any) continue;
#pragma unroll
      for (int c = 0; c < KM; ++c)
        if (c < K) acc[c * hw + p] = a[c];
      wsum[p] = ws;
    }
  } else {
    __shared__ float sz[KM][16][17];                   // [class][box row][box column] of one tile's logits
    const int lo = threadIdx.x & 15, hi = threadIdx.x >> 4;
    const int bxn = (bw + 15) / 16, n_box = ((bh + 15) / 16) * bxn;
    for (int q = blockIdx.x; q < n_box; q += gridDim.x) {             // uniform per CTA
      const int by0 = y0 + (q / bxn) * 16, bx0 = x0 + (q % bxn) * 16;
      const int Y = by0 + hi, X = bx0 + lo;                            // this thread's pixel
      PixelCover cv;
      const bool mine = Y < y0 + bh && X < x0 + bw && batch_cover(ay, ax, Y, X, t0, t1, cv);
      const bool fresh = mine && cv.fresh && first_pass;
      const long long p = static_cast<long long>(Y) * ax.len + X;
      float a[KM];
      float ws = 0.f;
#pragma unroll
      for (int c = 0; c < KM; ++c) a[c] = (mine && c < K && !fresh) ? acc[c * hw + p] : 0.f;
      if (mine && !fresh) ws = wsum[p];
      bool any = false;
      // the tiles that cover some pixel of the box: contiguous ranges per axis
      int tya, tyb, txa, txb, dummy;
      axis_cover(ay, by0, tya, dummy);
      axis_cover(ay, min(by0 + 15, ay.len - 1), dummy, tyb);
      axis_cover(ax, bx0, txa, dummy);
      axis_cover(ax, min(bx0 + 15, ax.len - 1), dummy, txb);
      // the copy: consecutive threads on consecutive rows of the box
      const int LY = by0 + lo, LX = bx0 + hi;
      for (int ty = tya; ty <= tyb; ++ty) {
        const int row = ty * ax.n;
        const int xa = max(txa, t0 - row), xb = min(txb, t1 - 1 - row);
        for (int tx = xa; tx <= xb; ++tx) {
          const int b = row + tx - t0;
          const int oy = axis_origin(ay, ty), ox = axis_origin(ax, tx);
          __syncthreads();                             // the previous tile's reads of sz are done
          if (LY < ay.len && LX < ax.len && LY >= oy && LY < oy + ay.ext && LX >= ox && LX < ox + ax.ext) {
            const float* lg = logits + b * K * tile_px + tta_offset(d, LY - oy, LX - ox, ay.ext, ax.ext);
#pragma unroll
            for (int c = 0; c < KM; ++c)
              if (c < K) sz[c][lo][hi] = __ldg(lg + c * tile_px);
          }
          __syncthreads();
          if (mine && Y >= oy && Y < oy + ay.ext && X >= ox && X < ox + ax.ext) {
            const float w = gy(Y - oy) * gx(X - ox);
            blend_tile<KT>([&](int c) { return sz[c][hi][lo]; }, K, w, a);
            ws += w;
            any = true;
          }
        }
      }
      if (!any) continue;
#pragma unroll
      for (int c = 0; c < KM; ++c)
        if (c < K) acc[c * hw + p] = a[c];
      wsum[p] = ws;
    }
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
  __shared__ unsigned int hist[kConfusionMaxBins];
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
      if (labels) bin = confusion_bin(labels[i], best, K, ignore);
    }
    if (labels) hist_add_warp(hist, bin);
  }
  if (labels) {
    __syncthreads();
    hist_flush(hist, bins, counts);
  }
}

// ------------------------------------------------------------------------------------------------
// Image blend (translate_scene), gather form like scene_blend_kernel and with the same tile-visit rule: one thread per
// scene pixel of the batch's box, consecutive threads on consecutive columns of one row (a 2-D grid-stride loop, so
// no 64-bit division per pixel).  Each covering tile of the batch costs one 16-byte load of the generator's 4-slot
// fp32 output and C + 1 FMAs.  The per-axis window is tabulated once per CTA in shared memory (ey + ex values of the
// same window()), so the per-pixel work has no exp.
// ------------------------------------------------------------------------------------------------
constexpr int kSceneMaxWindow = 12288;     // ey + ex: the window table fits the default 48 KB of dynamic shared memory

template <int C>
__global__ void __launch_bounds__(256) scene_blend_image_kernel(const float4* __restrict__ fake, SceneAxis ay,
                                                                SceneAxis ax, int t0, int t1, int y0, int x0, int bh,
                                                                int bw, float* __restrict__ acc,
                                                                float* __restrict__ wsum) {
  extern __shared__ float win[];           // g_y [ey], then g_x [ex]
  float* gy = win;
  float* gx = win + ay.ext;
  for (int i = threadIdx.x; i < ay.ext; i += blockDim.x) gy[i] = window(i, ay.ext);
  for (int i = threadIdx.x; i < ax.ext; i += blockDim.x) gx[i] = window(i, ax.ext);
  __syncthreads();
  const long long hw = static_cast<long long>(ay.len) * ax.len;
  const long long tile_px = static_cast<long long>(ay.ext) * ax.ext;
  for (int Y = y0 + blockIdx.y; Y < y0 + bh; Y += gridDim.y) {
    for (int X = x0 + blockIdx.x * blockDim.x + threadIdx.x; X < x0 + bw; X += gridDim.x * blockDim.x) {
      PixelCover cv;
      if (!batch_cover(ay, ax, Y, X, t0, t1, cv)) continue;
      const long long p = static_cast<long long>(Y) * ax.len + X;
      float a[C];
      float ws = 0.f;
#pragma unroll
      for (int c = 0; c < C; ++c) a[c] = cv.fresh ? 0.f : acc[c * hw + p];
      if (!cv.fresh) ws = wsum[p];
      const bool any = visit_batch_tiles(
          ay, ax, Y, X, t0, t1, cv, [gy](int d) { return gy[d]; }, [gx](int d) { return gx[d]; },
          [&](int b, int ty, int tx, float w) {
            const float4 v = __ldg(fake + b * tile_px + static_cast<long long>(ty) * ax.ext + tx);
            a[0] = fmaf(w, v.x, a[0]);
            if (C > 1) a[1] = fmaf(w, v.y, a[1]);
            if (C > 2) a[2] = fmaf(w, v.z, a[2]);
            if (C > 3) a[3] = fmaf(w, v.w, a[3]);
            ws += w;
          });
      if (!any) continue;
#pragma unroll
      for (int c = 0; c < C; ++c) acc[c * hw + p] = a[c];
      wsum[p] = ws;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Image finalize: v = acc / wsum per channel; image[pixel][c] = uint8(clamp((v*0.5 + 0.5)*255, 0, 255)), truncated
// (the rule of the generator's out_u8 epilogue in thin_layers.cu and of torchvision's to_pil_image); write_float: v
// overwrites acc.  VEC: four pixels per thread, 16-byte loads of wsum and of every plane, and one 4C-byte store of
// their interleaved image bytes (needs pixels % 4 == 0 and aligned buffers; the host picks it).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t image_u8(float v) {
  return static_cast<uint32_t>(static_cast<uint8_t>(fminf(fmaxf((v * 0.5f + 0.5f) * 255.f, 0.f), 255.f)));
}

template <int C, bool VEC>
__global__ void __launch_bounds__(256) scene_finalize_image_kernel(float* __restrict__ acc,
                                                                   const float* __restrict__ wsum, long long hw,
                                                                   uint8_t* __restrict__ image, int write_float) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  const long long start = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  if constexpr (!VEC) {
    for (long long i = start; i < hw; i += stride) {
      const float ws = wsum[i];
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const float v = acc[c * hw + i] / ws;
        if (write_float) acc[c * hw + i] = v;
        image[i * C + c] = static_cast<uint8_t>(image_u8(v));
      }
    }
  } else {
    for (long long g = start; g < hw / 4; g += stride) {
      const float4 ws = reinterpret_cast<const float4*>(wsum)[g];
      uint32_t word[C];                      // the 4C image bytes of the four pixels, pixel-major
#pragma unroll
      for (int j = 0; j < C; ++j) word[j] = 0u;
#pragma unroll
      for (int c = 0; c < C; ++c) {
        float4* pl = reinterpret_cast<float4*>(acc + c * hw) + g;
        float4 v = *pl;
        v.x = v.x / ws.x;
        v.y = v.y / ws.y;
        v.z = v.z / ws.z;
        v.w = v.w / ws.w;
        if (write_float) *pl = v;
        const float q[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int px = 0; px < 4; ++px) {
          const int k = px * C + c;
          word[k >> 2] |= image_u8(q[px]) << ((k & 3) * 8);
        }
      }
      uint8_t* o = image + g * 4 * C;
      if (C == 1) {
        *reinterpret_cast<uint32_t*>(o) = word[0];
      } else if (C == 2) {
        *reinterpret_cast<uint2*>(o) = make_uint2(word[0], word[C > 1 ? 1 : 0]);
      } else if (C == 3) {
#pragma unroll
        for (int j = 0; j < C; ++j) reinterpret_cast<uint32_t*>(o)[j] = word[j];
      } else {
        *reinterpret_cast<uint4*>(o) =
            make_uint4(word[0], word[C > 1 ? 1 : 0], word[C > 2 ? 2 : 0], word[C > 3 ? 3 : 0]);
      }
    }
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

// Tiles [t0, t1) of a batch and the box [y0, y0 + bh) x [x0, x0 + bw) they cover: their tile rows, and their columns
// when they share one tile row.
struct SceneBox {
  int t0, t1, y0, x0, bh, bw;
};

static inline SceneBox scene_batch_box(const SceneAxis& ay, const SceneAxis& ax, int tile0, int batch) {
  const int nx = ax.n;
  const int t0 = tile0, t1 = std::min(tile0 + batch, ay.n * nx);
  const int ty0 = t0 / nx, ty1 = (t1 - 1) / nx;
  const int y0 = scene_origin_host(ay, ty0), y1 = std::min(scene_origin_host(ay, ty1) + ay.ext, ay.len);
  int x0 = 0, x1 = ax.len;
  if (ty0 == ty1) {
    x0 = scene_origin_host(ax, t0 - ty0 * nx);
    x1 = std::min(scene_origin_host(ax, t1 - 1 - ty0 * nx) + ax.ext, ax.len);
  }
  return SceneBox{t0, t1, y0, x0, y1 - y0, x1 - x0};
}

template <int NIMG, bool S>
static void scene_gather_launch(const void* img1, const void* img2, int src_u8, int c, const SceneAxis& ay,
                                const SceneAxis& ax, int tile0, int batch, int d, void* out1, void* out2,
                                cudaStream_t st) {
  // one thread per output pixel, or (S) one CTA of 256 threads per 16 x 16 square: the same CTA count
  const int grid = scene_grid(static_cast<long long>(ay.ext) * ax.ext * batch, 148 * 8);
  bf16* o1 = static_cast<bf16*>(out1);
  bf16* o2 = static_cast<bf16*>(out2);
#define GATHER(CC, U) \
  scene_gather_kernel<CC, U, NIMG, S><<<grid, 256, 0, st>>>(img1, img2, ay, ax, tile0, batch, d, o1, o2)
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
}

}  // namespace gap

using namespace gap;

extern "C" {

int gap_scene_gather_tta(const void* img1, const void* img2, int src_u8, int c, int h, int w, int ey, int ex, int sy,
                         int sx, int ny, int nx, int tile0, int batch, int d, void* out1, void* out2, void* stream) {
  GAP_CHECK_ARG(c >= 1 && c <= 4, "gap_scene_gather: c must be 1..4, got %d", c);
  GAP_CHECK_ARG(d >= 0 && d <= 7, "gap_scene_gather: d must be 0..7, got %d", d);
  const SceneAxis ay{h, ey, sy, ny}, ax{w, ex, sx, nx};
  GAP_CHECK_ARG(img1 && img2 && out1 && out2 && scene_axis_ok(ay) && scene_axis_ok(ax) && batch >= 1 && tile0 >= 0 &&
                    tile0 < ny * nx,
                "gap_scene_gather: bad arguments");
  GAP_CHECK_ARG((reinterpret_cast<uintptr_t>(out1) & 7) == 0 && (reinterpret_cast<uintptr_t>(out2) & 7) == 0,
                "gap_scene_gather: out1 / out2 must be 8-byte aligned (one 8-byte store per 4-slot pixel)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (d & 4)
    scene_gather_launch<2, true>(img1, img2, src_u8, c, ay, ax, tile0, batch, d, out1, out2, st);
  else
    scene_gather_launch<2, false>(img1, img2, src_u8, c, ay, ax, tile0, batch, d, out1, out2, st);
  GAP_CUDA(cudaGetLastError());
  return 0;
}

int gap_scene_gather(const void* img1, const void* img2, int src_u8, int c, int h, int w, int ey, int ex, int sy,
                     int sx, int ny, int nx, int tile0, int batch, void* out1, void* out2, void* stream) {
  return gap_scene_gather_tta(img1, img2, src_u8, c, h, w, ey, ex, sy, sx, ny, nx, tile0, batch, 0, out1, out2, stream);
}

int gap_scene_blend_tta(const float* logits, int k, int h, int w, int ey, int ex, int sy, int sx, int ny, int nx,
                        int tile0, int batch, int d, int first_pass, float* acc, float* wsum, void* stream) {
  GAP_CHECK_ARG(k >= 1 && k <= kSceneMaxClasses, "gap_scene_blend: k must be 1..16, got %d", k);
  GAP_CHECK_ARG(d >= 0 && d <= 7, "gap_scene_blend: d must be 0..7, got %d", d);
  const SceneAxis ay{h, ey, sy, ny}, ax{w, ex, sx, nx};
  GAP_CHECK_ARG(logits && acc && wsum && scene_axis_ok(ay) && scene_axis_ok(ax) && batch >= 1 && tile0 >= 0 &&
                    tile0 < ny * nx,
                "gap_scene_blend: bad arguments");
  const SceneBox bx = scene_batch_box(ay, ax, tile0, batch);
  const int t0 = bx.t0, t1 = bx.t1, y0 = bx.y0, x0 = bx.x0, bh = bx.bh, bw = bx.bw;
  const int fp = first_pass ? 1 : 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (d & 4) {        // one CTA per 16 x 16 box of pixels
    const int grid = static_cast<int>(std::min<long long>(static_cast<long long>((bh + 15) / 16) * ((bw + 15) / 16),
                                                          148 * 8));
#define BLEND(KK, SS) \
  scene_blend_kernel<KK, SS><<<grid, 256, 0, st>>>(logits, k, ay, ax, t0, t1, y0, x0, bh, bw, d, fp, acc, wsum)
    switch (k) {
      case 1: BLEND(1, true); break;
      case 2: BLEND(2, true); break;
      default: BLEND(0, true); break;
    }
  } else {
    const int grid = scene_grid(static_cast<long long>(bh) * bw, 148 * 8);
    switch (k) {
      case 1: BLEND(1, false); break;
      case 2: BLEND(2, false); break;
      default: BLEND(0, false); break;
    }
#undef BLEND
  }
  GAP_CUDA(cudaGetLastError());
  return 0;
}

int gap_scene_blend(const float* logits, int k, int h, int w, int ey, int ex, int sy, int sx, int ny, int nx, int tile0,
                    int batch, float* acc, float* wsum, void* stream) {
  return gap_scene_blend_tta(logits, k, h, w, ey, ex, sy, sx, ny, nx, tile0, batch, 0, 1, acc, wsum, stream);
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

int gap_scene_gather_one(const void* img, int src_u8, int c, int h, int w, int ey, int ex, int sy, int sx, int ny,
                         int nx, int tile0, int batch, void* out, void* stream) {
  GAP_CHECK_ARG(c >= 1 && c <= 4, "gap_scene_gather_one: c must be 1..4, got %d", c);
  const SceneAxis ay{h, ey, sy, ny}, ax{w, ex, sx, nx};
  GAP_CHECK_ARG(img && out && scene_axis_ok(ay) && scene_axis_ok(ax) && batch >= 1 && tile0 >= 0 && tile0 < ny * nx,
                "gap_scene_gather_one: bad arguments");
  GAP_CHECK_ARG((reinterpret_cast<uintptr_t>(out) & 7) == 0,
                "gap_scene_gather_one: out must be 8-byte aligned (one 8-byte store per 4-slot pixel)");
  scene_gather_launch<1, false>(img, nullptr, src_u8, c, ay, ax, tile0, batch, 0, out, nullptr,
                                static_cast<cudaStream_t>(stream));
  GAP_CUDA(cudaGetLastError());
  return 0;
}

int gap_scene_blend_image(const float* fake, int c, int h, int w, int ey, int ex, int sy, int sx, int ny, int nx,
                          int tile0, int batch, float* acc, float* wsum, void* stream) {
  GAP_CHECK_ARG(c >= 1 && c <= 4, "gap_scene_blend_image: c must be 1..4, got %d", c);
  const SceneAxis ay{h, ey, sy, ny}, ax{w, ex, sx, nx};
  GAP_CHECK_ARG(fake && acc && wsum && scene_axis_ok(ay) && scene_axis_ok(ax) && batch >= 1 && tile0 >= 0 &&
                    tile0 < ny * nx,
                "gap_scene_blend_image: bad arguments");
  GAP_CHECK_ARG(ey + ex <= kSceneMaxWindow, "gap_scene_blend_image: ey + ex = %d exceeds %d", ey + ex, kSceneMaxWindow);
  GAP_CHECK_ARG((reinterpret_cast<uintptr_t>(fake) & 15) == 0,
                "gap_scene_blend_image: fake must be 16-byte aligned (one 16-byte load per 4-slot pixel)");
  const SceneBox bx = scene_batch_box(ay, ax, tile0, batch);
  const size_t smem = static_cast<size_t>(ey + ex) * sizeof(float);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const float4* f4 = reinterpret_cast<const float4*>(fake);
#define BLEND_IMG(CC)                                                                                              \
  do {                                                                                                             \
    int occ = 0;                                                                                                   \
    GAP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, scene_blend_image_kernel<CC>, 256, smem));        \
    const int blocks = 148 * std::max(occ, 1);                                                                     \
    const int gx = static_cast<int>(std::min<long long>((bx.bw + 255) / 256, blocks));                              \
    const int gy = std::max(1, std::min(bx.bh, std::min(blocks / gx, 65535)));                                     \
    scene_blend_image_kernel<CC><<<dim3(gx, gy), 256, smem, st>>>(f4, ay, ax, bx.t0, bx.t1, bx.y0, bx.x0, bx.bh,   \
                                                                  bx.bw, acc, wsum);                               \
  } while (0)
  switch (c) {
    case 1: BLEND_IMG(1); break;
    case 2: BLEND_IMG(2); break;
    case 3: BLEND_IMG(3); break;
    default: BLEND_IMG(4); break;
  }
#undef BLEND_IMG
  GAP_CUDA(cudaGetLastError());
  return 0;
}

int gap_scene_finalize_image(float* acc, const float* wsum, int c, int64_t pixels, uint8_t* image, int write_float,
                             void* stream) {
  GAP_CHECK_ARG(c >= 1 && c <= 4, "gap_scene_finalize_image: c must be 1..4, got %d", c);
  GAP_CHECK_ARG(acc && wsum && image && pixels > 0, "gap_scene_finalize_image: bad arguments");
  const uintptr_t img_align = c == 3 ? 4 : 4 * c;
  const bool vec = pixels % 4 == 0 && (reinterpret_cast<uintptr_t>(acc) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(wsum) & 15) == 0 && reinterpret_cast<uintptr_t>(image) % img_align == 0;
  const int grid = scene_grid(vec ? pixels / 4 : pixels, 148 * 8);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
#define FIN_IMG(CC)                                                                                                \
  do {                                                                                                             \
    if (vec)                                                                                                       \
      scene_finalize_image_kernel<CC, true><<<grid, 256, 0, st>>>(acc, wsum, pixels, image, write_float);          \
    else                                                                                                           \
      scene_finalize_image_kernel<CC, false><<<grid, 256, 0, st>>>(acc, wsum, pixels, image, write_float);         \
  } while (0)
  switch (c) {
    case 1: FIN_IMG(1); break;
    case 2: FIN_IMG(2); break;
    case 3: FIN_IMG(3); break;
    default: FIN_IMG(4); break;
  }
#undef FIN_IMG
  GAP_CUDA(cudaGetLastError());
  return 0;
}

}  // extern "C"
