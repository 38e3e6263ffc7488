// Change objects (objects.change_objects): connected-component labelling of a uint8 class map [n][h][w] (and, for
// the object-level scores, of the label map), minimum-area filtering, raster-order numbering and the object table.
//
// An object is a maximal 4- or 8-connected set of pixels of one non-zero class inside one sample.  The labelling is
// the block-based union-find of Playne & Hawick (IEEE TPDS 2018) / Allegretti et al. (IEEE TPDS 2019):
//   local    each CTA labels a 32 x 32 block in shared memory and writes, per pixel, the global raster index of its
//            block-local root;
//   border   threads on the block borders union across blocks in global memory;
//   flatten  every pixel's parent becomes its root, and each root's area is counted with integer atomics (one per
//            local root and block).
// Every union links the larger root under the smaller one (atomicMin, lock-free), so parent[i] <= i always holds and
// each root is its component's first pixel in raster order over (n, y, x), whatever the scheduling.  A device-wide
// exclusive scan over the keep flags of the roots (class != 0, area >= min_area; per-CTA counts, one CTA scanning
// those, then the numbering) gives the ids 1..count in raster order of the first pixel, as scipy.ndimage.label run per
// class and renumbered by first pixel would.  Only integer atomics are used: every output is bit-identical from run to
// run.
//
// gap_objects_label   class map (uint8 pred, or int64 labels -> uint8 label classes) -> parent (roots) and root areas
// gap_objects_number  roots + areas -> ids of the kept roots (in place of the areas) and the object count
// gap_objects_finish  ids of every pixel, filtered pred, confusion, overlaps, the object table and the object counts
#include <algorithm>

#include "common.h"
#include "confusion.cuh"

namespace gap {

constexpr int kObjBlock = 32;                     // side of the square block of the local labelling
constexpr int kObjChunk = 4096;                   // pixels per CTA of the numbering (256 threads x 16)
constexpr int kObjMaxClasses = 16;
constexpr int kObjNoLabel = 0xFF;                 // label class of an ignored or out-of-range label

// A pixel of class v joins objects unless it is background (0) or an uncounted label.
__device__ __forceinline__ bool obj_fg(int v) { return v != 0 && v != kObjNoLabel; }

// Pixels of the reduction needed for a match: max(1, ceil(min_overlap * area)), formed in fp64.
__device__ __forceinline__ long long obj_needed(long long area, double min_overlap) {
  const long long t = static_cast<long long>(ceil(min_overlap * static_cast<double>(area)));
  return t < 1 ? 1 : t;
}

// Block (s, by, bx) of CTA blockIdx.x, numbered row-major over [n][ceil(h/32)][ceil(w/32)].
__device__ __forceinline__ void obj_block(int h, int w, int& s, int& y0, int& x0) {
  const int bxn = (w + kObjBlock - 1) / kObjBlock, byn = (h + kObjBlock - 1) / kObjBlock;
  int b = blockIdx.x;
  const int bx = b % bxn;
  b /= bxn;
  const int by = b % byn;
  s = b / byn;
  y0 = by * kObjBlock;
  x0 = bx * kObjBlock;
}

// ---- union-find: parent[a] <= a, roots are minima; a union links the larger root under the smaller ----
__device__ __forceinline__ int local_find(const volatile int* par, int a) {
  int p = par[a];
  while (p != a) {
    a = p;
    p = par[a];
  }
  return a;
}

__device__ __forceinline__ void local_union(int* par, int a, int b) {
  while (true) {
    a = local_find(par, a);
    b = local_find(par, b);
    if (a == b) return;
    if (a < b) {
      const int t = a;
      a = b;
      b = t;
    }
    const int old = atomicMin(par + a, b);
    if (old == a) return;
    a = old;                                       // a was linked elsewhere meanwhile: join that tree to b instead
  }
}

__device__ __forceinline__ int global_find(const int* par, int a) {
  int p = __ldcg(par + a);
  while (p != a) {
    a = p;
    p = __ldcg(par + a);
  }
  return a;
}

__device__ __forceinline__ void global_union(int* par, int a, int b) {
  while (true) {
    a = global_find(par, a);
    b = global_find(par, b);
    if (a == b) return;
    if (a < b) {
      const int t = a;
      a = b;
      b = t;
    }
    const int old = atomicMin(par + a, b);
    if (old == a) return;
    a = old;
  }
}

// ------------------------------------------------------------------------------------------------
// Local labelling: one 32 x 32 block per CTA, 256 threads, each on one column and four rows (ly, ly + 8, ...).
// LABELS: src is int64 labels; the label class (kObjNoLabel for ignore_index and values outside [0, kk)) is written to
// classes.  Otherwise src is the uint8 pred and values >= kk are counted into *bad.  Pixels outside the scene are
// background in shared memory, so unions need no bounds checks.
// ------------------------------------------------------------------------------------------------
template <bool LABELS>
__global__ void __launch_bounds__(256) objects_local_kernel(const void* __restrict__ src, int h, int w, int kk,
                                                            long long ignore, int conn8, uint8_t* __restrict__ classes,
                                                            int* __restrict__ parent, int* __restrict__ bad) {
  __shared__ int par[kObjBlock * kObjBlock];
  __shared__ uint8_t cl[kObjBlock * kObjBlock];
  int s, y0, x0;
  obj_block(h, w, s, y0, x0);
  const int lx = threadIdx.x & 31, x = x0 + lx;
  int nbad = 0;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int ly = (threadIdx.x >> 5) + 8 * j, y = y0 + ly, l = ly * kObjBlock + lx;
    int v = 0;
    if (x < w && y < h) {
      const int i = (s * h + y) * w + x;
      if (LABELS) {
        const long long yv = static_cast<const long long*>(src)[i];
        v = (yv != ignore && yv >= 0 && yv < kk) ? static_cast<int>(yv) : kObjNoLabel;
        classes[i] = static_cast<uint8_t>(v);
      } else {
        v = static_cast<const uint8_t*>(src)[i];
        nbad += v >= kk;
      }
    }
    cl[l] = static_cast<uint8_t>(v);
    par[l] = l;
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int ly = (threadIdx.x >> 5) + 8 * j, l = ly * kObjBlock + lx;
    const int v = cl[l];
    if (!obj_fg(v)) continue;
    if (lx > 0 && cl[l - 1] == v) local_union(par, l, l - 1);
    if (ly > 0) {
      const int u = l - kObjBlock;
      if (cl[u] == v) local_union(par, l, u);
      if (conn8 && lx > 0 && cl[u - 1] == v) local_union(par, l, u - 1);
      if (conn8 && lx < kObjBlock - 1 && cl[u + 1] == v) local_union(par, l, u + 1);
    }
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int ly = (threadIdx.x >> 5) + 8 * j, y = y0 + ly, l = ly * kObjBlock + lx;
    if (x >= w || y >= h) continue;
    const int r = local_find(par, l);
    parent[(s * h + y) * w + x] = (s * h + y0 + r / kObjBlock) * w + x0 + r % kObjBlock;
  }
  if (!LABELS) {
    nbad = __reduce_add_sync(0xffffffffu, nbad);
    if (nbad && lx == 0) atomicAdd(bad, nbad);
  }
}

// ------------------------------------------------------------------------------------------------
// Border merge: per block, 96 threads.  Every pair of adjacent pixels is joined from its later pixel (in raster order)
// towards the earlier one; this kernel handles the pairs whose two pixels lie in different blocks of one sample:
//   threads  0..31  the top row: the pixels above (and, 8-connected, above-left / above-right) in the block row above
//   threads 32..63  the left column: the pixel to the left (and, 8-connected and below the top row, above-left)
//   threads 64..95  the right column below the top row, 8-connected: the pixel above-right, in the block to the right
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(96) objects_border_kernel(const uint8_t* __restrict__ cls, int h, int w, int conn8,
                                                            int* __restrict__ parent) {
  int s, y0, x0;
  obj_block(h, w, s, y0, x0);
  const int t = threadIdx.x;
  int y, x;
  if (t < 32) {
    if (y0 == 0) return;
    y = y0;
    x = x0 + t;
  } else if (t < 64) {
    if (x0 == 0) return;
    y = y0 + t - 32;
    x = x0;
  } else {
    if (!conn8 || t == 64 || x0 + kObjBlock >= w) return;
    y = y0 + t - 64;
    x = x0 + kObjBlock - 1;
  }
  if (x >= w || y >= h) return;
  const int i = (s * h + y) * w + x;
  const int v = cls[i];
  if (!obj_fg(v)) return;
  auto join = [&](int q) {
    if (cls[q] == v) global_union(parent, i, q);
  };
  if (t < 32) {
    join(i - w);
    if (conn8 && x > 0) join(i - w - 1);
    if (conn8 && x + 1 < w) join(i - w + 1);
  } else if (t < 64) {
    join(i - 1);
    if (conn8 && y > y0) join(i - w - 1);
  } else {
    join(i - w + 1);
  }
}

// ------------------------------------------------------------------------------------------------
// Flatten, per 32 x 32 block like the local labelling: parent[i] = root of i, and area[root] += 1 for every object
// pixel.  A pixel whose parent lies in its block points at its local root (local parents are never changed by the
// border merge); a pixel whose parent lies elsewhere is a local root the border merge linked.  The pixels of a local
// root are counted in shared memory, then one thread per local root walks the global tree once and adds the count at
// the final root, so a component that spans many blocks costs one walk and one atomic per block, not per pixel.  The
// forest no longer changes here, so plain (L1-cached) loads see valid ancestors.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) objects_flatten_kernel(const uint8_t* __restrict__ cls, int h, int w,
                                                              int* __restrict__ parent, int* __restrict__ area) {
  __shared__ int cnt[kObjBlock * kObjBlock];
  __shared__ int root[kObjBlock * kObjBlock];
  int s, y0, x0;
  obj_block(h, w, s, y0, x0);
  const int lx = threadIdx.x & 31, x = x0 + lx;
  const int row0 = s * h + y0;                        // global row of the block's first row
  int lp[4], pp[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) cnt[((threadIdx.x >> 5) + 8 * j) * kObjBlock + lx] = 0;
  __syncthreads();
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int ly = (threadIdx.x >> 5) + 8 * j, y = y0 + ly, l = ly * kObjBlock + lx;
    lp[j] = -1;
    if (x >= w || y >= h) continue;
    const int i = (row0 + ly) * w + x;
    if (!obj_fg(cls[i])) continue;
    const int p = parent[i];
    pp[j] = p;
    const int py = p / w - row0, px = p % w - x0;
    lp[j] = (py >= 0 && py < kObjBlock && px >= 0 && px < kObjBlock) ? py * kObjBlock + px : l;
    atomicAdd(&cnt[lp[j]], 1);
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int ly = (threadIdx.x >> 5) + 8 * j, l = ly * kObjBlock + lx;
    const int c = cnt[l];
    if (c == 0) continue;
    int r = (row0 + ly) * w + x;
    for (int q = parent[r]; q != r; q = parent[r]) r = q;
    root[l] = r;
    atomicAdd(area + r, c);
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (lp[j] < 0) continue;
    const int r = root[lp[j]];
    if (r != pp[j]) parent[(row0 + (threadIdx.x >> 5) + 8 * j) * w + x] = r;
  }
}

// ------------------------------------------------------------------------------------------------
// Numbering: a root is kept when its class is non-zero and its area >= min_area.  count: kept roots per chunk of
// kObjChunk pixels; scan: one CTA turns the chunk counts into exclusive offsets and writes the total to info[0];
// number: area_ids[root] = its id (1 + kept roots before it in raster order) or 0 when it is dropped.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) objects_count_kernel(const uint8_t* __restrict__ cls,
                                                            const int* __restrict__ parent,
                                                            const int* __restrict__ area, long long total,
                                                            long long min_area, int* __restrict__ chunk) {
  __shared__ int wsum[8];
  const long long base = static_cast<long long>(blockIdx.x) * kObjChunk;
  int c = 0;
#pragma unroll 4
  for (int j = 0; j < kObjChunk / 256; ++j) {
    const long long i = base + j * 256 + threadIdx.x;
    if (i < total && parent[i] == i && obj_fg(cls[i]) && area[i] >= min_area) ++c;
  }
  c = __reduce_add_sync(0xffffffffu, c);
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    int s = 0;
    for (int k = 0; k < 8; ++k) s += wsum[k];
    chunk[blockIdx.x] = s;
  }
}

__global__ void __launch_bounds__(1024) objects_scan_kernel(int* __restrict__ chunk, int nchunks, int* __restrict__ info) {
  __shared__ int wsum[32];
  const int per = (nchunks + 1023) / 1024;
  const int a = min(static_cast<int>(threadIdx.x) * per, nchunks), b = min(a + per, nchunks);
  int s = 0;
  for (int k = a; k < b; ++k) s += chunk[k];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = s;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int u = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += u;
  }
  if (lane == 31) wsum[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int v = wsum[lane];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, v, d);
      if (lane >= d) v += u;
    }
    wsum[lane] = v;                                 // inclusive sums of the warps
  }
  __syncthreads();
  int run = incl - s + (warp > 0 ? wsum[warp - 1] : 0);
  for (int k = a; k < b; ++k) {
    const int c = chunk[k];
    chunk[k] = run;
    run += c;
  }
  if (threadIdx.x == 1023) info[0] = wsum[31];
}

__global__ void __launch_bounds__(256) objects_number_kernel(const uint8_t* __restrict__ cls,
                                                             const int* __restrict__ parent, int* __restrict__ area_ids,
                                                             long long total, long long min_area,
                                                             const int* __restrict__ chunk) {
  __shared__ int wsum[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long base = static_cast<long long>(blockIdx.x) * kObjChunk;
  int run = chunk[blockIdx.x];
  for (int j = 0; j < kObjChunk / 256; ++j) {
    const long long i = base + j * 256 + threadIdx.x;
    bool root = false, keep = false;
    if (i < total && parent[i] == i && obj_fg(cls[i])) {
      root = true;
      keep = area_ids[i] >= min_area;
    }
    const unsigned int kb = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) wsum[warp] = __popc(kb);
    __syncthreads();
    int before = 0, all = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      before += k < warp ? wsum[k] : 0;
      all += wsum[k];
    }
    if (root) area_ids[i] = keep ? run + before + __popc(kb & ((1u << lane) - 1u)) + 1 : 0;
    run += all;
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// After the count is known.
// init: object rows (area 0, x0 = +inf, y1 = x1 = -1; sample, class and y0 come from the first pixel) and overlaps.
// apply: ids of every pixel, the filtered pred, and with labels (whose classes arrive in pred_out) the confusion
//   histogram and the overlap pixels (filtered pred == label class != 0) of the predicted and the reference objects.
//   A reference root then stores -1 - class in its parent slot (no other pixel reads a root's slot after flatten).
// table: box and area atomics per object, warp-aggregated; reference objects counted (and detected) per class.
// counts: predicted (and matched) objects per class.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) objects_init_kernel(long long count, long long* __restrict__ objects,
                                                           int* __restrict__ overlap) {
  for (long long o = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; o < count;
       o += static_cast<long long>(gridDim.x) * blockDim.x) {
    long long* r = objects + o * 7;
    r[2] = 0;
    r[4] = 0x7fffffffffffffffLL;
    r[5] = -1;
    r[6] = -1;
    if (overlap) overlap[o] = 0;
  }
}

__global__ void __launch_bounds__(256) objects_apply_kernel(const uint8_t* __restrict__ pred,
                                                            const int* __restrict__ parent, int* __restrict__ ids,
                                                            long long total, int k, int kk,
                                                            uint8_t* __restrict__ pred_out, int* __restrict__ lparent,
                                                            int* __restrict__ loverlap, int* __restrict__ overlap,
                                                            unsigned long long* __restrict__ confusion) {
  __shared__ unsigned int hist[kConfusionMaxBins];
  const bool labels = lparent != nullptr;
  const int bins = k == 1 ? 4 : k * k;
  if (labels) {
    for (int i = threadIdx.x; i < bins; i += blockDim.x) hist[i] = 0u;
    __syncthreads();
  }
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i0 = blockIdx.x * static_cast<long long>(blockDim.x); i0 < total; i0 += stride) {   // uniform per warp
    const long long i = i0 + threadIdx.x;
    int bin = -1, okey = 0, rkey = -1;
    if (i < total) {
      const int p = parent[i];
      const int id = ids[p];
      if (p != i) ids[i] = id;
      const int f = id ? pred[i] : 0;
      if (labels) {
        const int lv = pred_out[i];
        const int lp = lparent[i];
        if (f < kk) bin = confusion_bin(lv == kObjNoLabel ? -1 : lv, f, k, -1);
        if (f != 0 && lv == f) {
          okey = id;
          rkey = lp;
        }
        if (lp == i && obj_fg(lv)) lparent[i] = -1 - lv;
      }
      pred_out[i] = static_cast<uint8_t>(f);
    }
    if (labels) {
      hist_add_warp(hist, bin);
      unsigned int peers = __match_any_sync(0xffffffffu, okey);
      if (okey > 0 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(overlap + okey - 1, __popc(peers));
      peers = __match_any_sync(0xffffffffu, rkey);
      if (rkey >= 0 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(loverlap + rkey, __popc(peers));
    }
  }
  if (labels) {
    __syncthreads();
    hist_flush(hist, bins, confusion);
  }
}

__global__ void __launch_bounds__(256) objects_table_kernel(const uint8_t* __restrict__ pred,
                                                            const int* __restrict__ parent, const int* __restrict__ ids,
                                                            int h, int w, long long total, long long* __restrict__ objects,
                                                            const int* __restrict__ lparent, const int* __restrict__ larea,
                                                            const int* __restrict__ loverlap, double min_overlap,
                                                            int kk, unsigned long long* __restrict__ ocounts) {
  __shared__ unsigned int hist[2 * kObjMaxClasses];     // per class: reference objects, detected ones
  const bool labels = lparent != nullptr;
  if (labels) {
    for (int i = threadIdx.x; i < 2 * kObjMaxClasses; i += blockDim.x) hist[i] = 0u;
    __syncthreads();
  }
  const int hw = h * w;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i0 = blockIdx.x * static_cast<long long>(blockDim.x); i0 < total; i0 += stride) {   // uniform per warp
    const long long i = i0 + threadIdx.x;
    int id = 0, x = 0, y = 0, ref = -1, det = -1;
    if (i < total) {
      id = ids[i];
      const int s = static_cast<int>(i / hw), r = static_cast<int>(i - static_cast<long long>(s) * hw);
      y = r / w;
      x = r - y * w;
      if (id > 0 && parent[i] == i) {                    // the object's first pixel
        long long* o = objects + static_cast<long long>(id - 1) * 7;
        o[0] = s;
        o[1] = pred[i];
        o[3] = y;
      }
      if (labels) {
        const int v = lparent[i];
        if (v < 0 && -1 - v < kk) {
          ref = 2 * (-1 - v);
          if (loverlap[i] >= obj_needed(larea[i], min_overlap)) det = ref + 1;
        }
      }
    }
    const unsigned int peers = __match_any_sync(0xffffffffu, id);
    if (id > 0) {
      const int xa = __reduce_min_sync(peers, x), xb = __reduce_max_sync(peers, x), yb = __reduce_max_sync(peers, y);
      if ((threadIdx.x & 31) == __ffs(peers) - 1) {
        long long* o = objects + static_cast<long long>(id - 1) * 7;
        atomicAdd(reinterpret_cast<unsigned long long*>(o + 2), static_cast<unsigned long long>(__popc(peers)));
        atomicMin(o + 4, static_cast<long long>(xa));
        atomicMax(o + 5, static_cast<long long>(yb));
        atomicMax(o + 6, static_cast<long long>(xb));
      }
    }
    if (labels) {
      hist_add_warp(hist, ref);
      hist_add_warp(hist, det);
    }
  }
  if (labels) {
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * kObjMaxClasses; i += blockDim.x)
      if (hist[i]) atomicAdd(ocounts + (i >> 1) * 4 + (i & 1), static_cast<unsigned long long>(hist[i]));
  }
}

__global__ void __launch_bounds__(256) objects_counts_kernel(const long long* __restrict__ objects,
                                                             const int* __restrict__ overlap, long long count,
                                                             double min_overlap, int kk,
                                                             unsigned long long* __restrict__ ocounts) {
  __shared__ unsigned int hist[2 * kObjMaxClasses];     // per class: predicted objects, matched ones
  for (int i = threadIdx.x; i < 2 * kObjMaxClasses; i += blockDim.x) hist[i] = 0u;
  __syncthreads();
  for (long long o = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; o < count;
       o += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long c = objects[o * 7 + 1];
    if (c < kk) {
      atomicAdd(&hist[2 * c], 1u);
      if (overlap[o] >= obj_needed(objects[o * 7 + 2], min_overlap)) atomicAdd(&hist[2 * c + 1], 1u);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * kObjMaxClasses; i += blockDim.x)
    if (hist[i]) atomicAdd(ocounts + (i >> 1) * 4 + 2 + (i & 1), static_cast<unsigned long long>(hist[i]));
}

static inline int objects_grid(long long work) {
  const long long g = std::max<long long>((work + 255) / 256, 1);
  return static_cast<int>(std::min<long long>(g, 148 * 8));
}

static inline bool objects_shape_ok(int n, int h, int w) {
  return n >= 1 && h >= 1 && w >= 1 && static_cast<long long>(n) * h * w < (1LL << 31);
}

}  // namespace gap

using namespace gap;

extern "C" {

int gap_objects_label(const void* src, int src_i64, int n, int h, int w, int k, int64_t ignore_index,
                      int connectivity, uint8_t* classes, int32_t* parent, int32_t* area, int32_t* info, void* stream) {
  GAP_CHECK_ARG(k >= 1 && k <= kObjMaxClasses, "gap_objects_label: k must be 1..16, got %d", k);
  GAP_CHECK_ARG(connectivity == 4 || connectivity == 8, "gap_objects_label: connectivity must be 4 or 8, got %d",
                connectivity);
  GAP_CHECK_ARG(objects_shape_ok(n, h, w), "gap_objects_label: need n, h, w >= 1 and n*h*w < 2^31, got %d x %d x %d",
                n, h, w);
  GAP_CHECK_ARG(src && parent && area && (src_i64 ? classes != nullptr : classes == nullptr && info != nullptr),
                "gap_objects_label: bad arguments");
  const long long total = static_cast<long long>(n) * h * w;
  const int kk = std::max(k, 2);
  const int conn8 = connectivity == 8;
  const long long blocks = static_cast<long long>(n) * ((h + kObjBlock - 1) / kObjBlock) * ((w + kObjBlock - 1) / kObjBlock);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  GAP_CUDA(cudaMemsetAsync(area, 0, total * sizeof(int32_t), st));
  const uint8_t* cls;
  if (src_i64) {
    objects_local_kernel<true><<<static_cast<unsigned>(blocks), 256, 0, st>>>(src, h, w, kk, ignore_index, conn8,
                                                                              classes, parent, nullptr);
    cls = classes;
  } else {
    GAP_CUDA(cudaMemsetAsync(info, 0, 2 * sizeof(int32_t), st));
    objects_local_kernel<false><<<static_cast<unsigned>(blocks), 256, 0, st>>>(src, h, w, kk, ignore_index, conn8,
                                                                               nullptr, parent, info + 1);
    cls = static_cast<const uint8_t*>(src);
  }
  objects_border_kernel<<<static_cast<unsigned>(blocks), 96, 0, st>>>(cls, h, w, conn8, parent);
  objects_flatten_kernel<<<static_cast<unsigned>(blocks), 256, 0, st>>>(cls, h, w, parent, area);
  GAP_CUDA(cudaGetLastError());
  return 0;
}

int gap_objects_number(const uint8_t* pred, const int32_t* parent, int32_t* area_ids, int64_t pixels, int64_t min_area,
                       int32_t* chunk, int32_t* info, void* stream) {
  GAP_CHECK_ARG(pred && parent && area_ids && chunk && info && pixels >= 1 && pixels < (1LL << 31) && min_area >= 0,
                "gap_objects_number: bad arguments");
  const long long nchunks = (pixels + kObjChunk - 1) / kObjChunk;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  objects_count_kernel<<<static_cast<unsigned>(nchunks), 256, 0, st>>>(pred, parent, area_ids, pixels, min_area, chunk);
  objects_scan_kernel<<<1, 1024, 0, st>>>(chunk, static_cast<int>(nchunks), info);
  objects_number_kernel<<<static_cast<unsigned>(nchunks), 256, 0, st>>>(pred, parent, area_ids, pixels, min_area, chunk);
  GAP_CUDA(cudaGetLastError());
  return 0;
}

int gap_objects_finish(const uint8_t* pred, const int32_t* parent, int32_t* ids, int n, int h, int w, int k,
                       int64_t count, uint8_t* pred_out, int32_t* overlap, int64_t* objects, int32_t* lparent,
                       const int32_t* larea, int32_t* loverlap, double min_overlap, int64_t* confusion,
                       int64_t* object_counts, void* stream) {
  GAP_CHECK_ARG(k >= 1 && k <= kObjMaxClasses, "gap_objects_finish: k must be 1..16, got %d", k);
  GAP_CHECK_ARG(objects_shape_ok(n, h, w), "gap_objects_finish: need n, h, w >= 1 and n*h*w < 2^31, got %d x %d x %d",
                n, h, w);
  const long long total = static_cast<long long>(n) * h * w;
  const bool labels = lparent != nullptr;
  GAP_CHECK_ARG(pred && parent && ids && pred_out && count >= 0 && count <= total && (count == 0 || objects),
                "gap_objects_finish: bad arguments");
  GAP_CHECK_ARG(labels ? larea && loverlap && confusion && object_counts && (count == 0 || overlap)
                       : !larea && !loverlap && !confusion && !object_counts,
                "gap_objects_finish: lparent, larea, loverlap, confusion and object_counts go together");
  GAP_CHECK_ARG(min_overlap >= 0.0 && min_overlap <= 1.0, "gap_objects_finish: min_overlap must be in [0, 1]");
  const int kk = std::max(k, 2);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned long long* conf = reinterpret_cast<unsigned long long*>(confusion);
  unsigned long long* oc = reinterpret_cast<unsigned long long*>(object_counts);
  long long* obj = reinterpret_cast<long long*>(objects);
  if (labels) {
    GAP_CUDA(cudaMemsetAsync(loverlap, 0, total * sizeof(int32_t), st));
    GAP_CUDA(cudaMemsetAsync(confusion, 0, (k == 1 ? 4 : k * k) * sizeof(int64_t), st));
    GAP_CUDA(cudaMemsetAsync(object_counts, 0, kk * 4 * sizeof(int64_t), st));
  }
  if (count > 0) objects_init_kernel<<<objects_grid(count), 256, 0, st>>>(count, obj, labels ? overlap : nullptr);
  const int grid = objects_grid(total);
  objects_apply_kernel<<<grid, 256, 0, st>>>(pred, parent, ids, total, k, kk, pred_out, lparent, loverlap,
                                             labels ? overlap : nullptr, conf);
  objects_table_kernel<<<grid, 256, 0, st>>>(pred, parent, ids, h, w, total, obj, lparent, larea, loverlap,
                                             min_overlap, kk, oc);
  if (labels && count > 0)
    objects_counts_kernel<<<objects_grid(count), 256, 0, st>>>(obj, overlap, count, min_overlap, kk, oc);
  GAP_CUDA(cudaGetLastError());
  return 0;
}

}  // extern "C"
