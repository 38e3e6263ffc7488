// Confusion counting shared by the scene finalize (scene.cu) and the change-object pass (objects.cu): the rule that
// maps a (label, prediction) pair to a bin, and the per-CTA shared-memory histogram those bins are added to.
#pragma once
#include <stdint.h>

namespace gap {

constexpr int kConfusionMaxBins = 16 * 16;

// The bin of one pixel, or -1 when it is not counted: k > 1 -> label * k + pred (rows = label); k = 1 -> [TP, FP, FN,
// TN] with label 1 positive and 0 negative.  Labels equal to ignore or outside [0, k) ({0, 1} for k = 1) are skipped.
__device__ __forceinline__ int confusion_bin(long long y, int pred, int k, long long ignore) {
  if (y == ignore || y < 0 || y >= (k == 1 ? 2 : k)) return -1;
  return k == 1 ? (y == 1 ? (pred ? 0 : 2) : (pred ? 1 : 3)) : static_cast<int>(y) * k + pred;
}

// Adds one bin per lane (bin < 0: nothing) to a shared-memory histogram; the lanes of a warp that share a bin add once.
// Every lane of the warp must call it.
__device__ __forceinline__ void hist_add_warp(unsigned int* hist, int bin) {
  const unsigned int peers = __match_any_sync(0xffffffffu, bin);
  if (bin >= 0 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&hist[bin], __popc(peers));
}

// Adds a CTA's histogram to the global counts (one 64-bit atomic per non-empty bin); call after a __syncthreads.
__device__ __forceinline__ void hist_flush(const unsigned int* hist, int bins, unsigned long long* counts) {
  for (int i = threadIdx.x; i < bins; i += blockDim.x)
    if (hist[i]) atomicAdd(counts + i, static_cast<unsigned long long>(hist[i]));
}

}  // namespace gap
