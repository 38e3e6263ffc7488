// Direct kernels for the HBM-bound "thin" layers of the PatchGAN discriminator and the U-Net
// generator: layers whose input or output has 1-6 channels move hundreds of MB for a few GFLOP, so
// they are fused, coalesced, warp-MMA (mma.sync) kernels that touch each activation once instead of
// im2col / channel-padded tcgen05 GEMMs.
//
//   gap_cout1_conv_{fwd,dgrad,wgrad}: Conv2d(C -> 1, k4, s1, p1) + bias, the discriminator's last layer
//   (models.py:243) and its two gradients.
#include "common.h"
#include "mma_sync.cuh"
#include "ptx.cuh"

namespace gap {

typedef __nv_bfloat16 bf16;

__device__ __forceinline__ uint4 ldg128(const void* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }
// 8-byte asynchronous global -> shared copy; src_bytes = 0 zero-fills the destination.
__device__ __forceinline__ void cp_async8(uint32_t dst, const void* src, int src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// ------------------------------------------------------------------------------------------------
// Cout = 1 forward, stage 1: z[pix][tap] = sum_c x[pix][c] * w[tap][c] for the 16 taps of a 4x4
// filter — every input element is read once (the 16 shifted sums are formed in stage 2 from z).
// CTA = 128 pixels, warp = 16 pixels x 16 taps, K = channels in chunks of 64.
// ------------------------------------------------------------------------------------------------
// PRE: the input is the raw (pre-BatchNorm) conv output y of the layer below and x = LeakyReLU(y*scale + shift) is
// formed while staging it (training-mode BatchNorm apply fused into the consumer: the activated tensor never exists
// in HBM).  The next 64-channel chunk's global loads are issued before the current chunk's MMAs.
struct Cout1Pre {
  const float* scale;
  const float* shift;
  float slope;
};

// eight consecutive fp32 parameters (32-byte aligned shared memory) as two 128-bit loads
__device__ __forceinline__ void lds8(const float* p, float (&r)[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  r[0] = a.x; r[1] = a.y; r[2] = a.z; r[3] = a.w;
  r[4] = b.x; r[5] = b.y; r[6] = b.z; r[7] = b.w;
}

// y*scale + shift, then x > 0 ? x : slope*x, on eight packed bf16 channels
__device__ __forceinline__ uint4 bn_act8(uint4 v, const float (&sc)[8], const float (&sh)[8], float slope) {
  uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float a = fmaf(bf16_lo(w[j]), sc[2 * j], sh[2 * j]);
    float b = fmaf(bf16_hi(w[j]), sc[2 * j + 1], sh[2 * j + 1]);
    a = a > 0.f ? a : slope * a;
    b = b > 0.f ? b : slope * b;
    w[j] = pack_bf16x2(a, b);
  }
  return make_uint4(w[0], w[1], w[2], w[3]);
}

template <bool PRE>
__global__ void __launch_bounds__(256, 4) cout1_z_kernel(const bf16* __restrict__ x, long long ld_x, long long npix,
                                                      int c, const bf16* __restrict__ w, float* __restrict__ z,
                                                      const Cout1Pre pre) {
  __shared__ __align__(16) bf16 xs[128][72];
  __shared__ __align__(16) bf16 ws[16][72];
  __shared__ __align__(16) float par[PRE ? 1024 : 4];   // scale[512] | shift[512]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t xs_a = smem_u32(&xs[0][0]), ws_a = smem_u32(&ws[0][0]);
  if (PRE) {
    for (int i = tid; i < c; i += 256) {
      par[i] = __ldg(pre.scale + i);
      par[512 + i] = __ldg(pre.shift + i);
    }
    __syncthreads();
  }
  for (long long tile = blockIdx.x; tile * 128 < npix; tile += gridDim.x) {
    float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
    uint4 nxt[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int v = tid + i * 256, px = v >> 3, seg = v & 7;
      const long long pix = tile * 128 + px;
      nxt[i] = pix < npix ? ldg128(x + pix * ld_x + seg * 8) : make_uint4(0, 0, 0, 0);
    }
    for (int c0 = 0; c0 < c; c0 += 64) {
      float sc[8], sh[8];       // this thread always stages the same 8 channels of a chunk (seg = tid & 7)
      if (PRE) {
        lds8(par + c0 + (tid & 7) * 8, sc);
        lds8(par + 512 + c0 + (tid & 7) * 8, sh);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int v = tid + i * 256, px = v >> 3, seg = v & 7;
        uint4 val = nxt[i];
        if (PRE && tile * 128 + px < npix) val = bn_act8(val, sc, sh, pre.slope);
        *reinterpret_cast<uint4*>(&xs[px][seg * 8]) = val;
      }
      if (tid < 128) {
        const int t = tid >> 3, seg = tid & 7;
        *reinterpret_cast<uint4*>(&ws[t][seg * 8]) = ldg128(w + static_cast<long long>(t) * c + c0 + seg * 8);
      }
      __syncthreads();
      if (c0 + 64 < c) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int v = tid + i * 256, px = v >> 3, seg = v & 7;
          const long long pix = tile * 128 + px;
          nxt[i] = pix < npix ? ldg128(x + pix * ld_x + c0 + 64 + seg * 8) : make_uint4(0, 0, 0, 0);
        }
      }
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        uint32_t a[4], b[4];
        lda_16x16(a, xs_a + warp * 16 * 144 + ks * 32, 144, lane);
        ldb_16x16(b, ws_a + ks * 32, 144, lane);
        mma_bf16_16816(acc[0], a, b[0], b[1]);
        mma_bf16_16816(acc[1], a, b[2], b[3]);
      }
      __syncthreads();
    }
    const int g = lane >> 2, t = lane & 3;
    const long long row0 = tile * 128 + warp * 16 + g, row1 = row0 + 8;
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) {
      if (row0 < npix) *reinterpret_cast<float2*>(z + row0 * 16 + nt * 8 + 2 * t) = make_float2(acc[nt][0], acc[nt][1]);
      if (row1 < npix) *reinterpret_cast<float2*>(z + row1 * 16 + nt * 8 + 2 * t) = make_float2(acc[nt][2], acc[nt][3]);
    }
  }
}

// stage 2: logits[n][oy][ox] = bias + sum_{kh,kw} z[n][oy+kh-pad][ox+kw-pad][kh*4+kw]
// Four adjacent lanes per output, one kernel row each (its four loads are issued together, then two shuffles): the
// one-thread-per-output loop with 16 conditional loads was latency-bound (6.9 us for 57600 outputs, ncu).
__global__ void __launch_bounds__(256) cout1_gather_kernel(const float* __restrict__ z, const float* __restrict__ bias, int n,
                                                           int ih, int iw, int oh, int ow, int pad,
                                                           float* __restrict__ logits) {
  const long long total = static_cast<long long>(n) * oh * ow;
  const long long groups = (total + 63) / 64;      // 64 outputs per block pass; every lane of a warp stays in the loop
  for (long long gi = blockIdx.x; gi < groups; gi += gridDim.x) {
    const long long i = gi * 64 + (threadIdx.x >> 2);
    const int kh = threadIdx.x & 3;
    float s = 0.f;
    if (i < total) {
      long long img;
      int ox, oy;
      if (total <= 0x7fffffffLL) {      // 32-bit divisions (the 64-bit ones are ~100 instructions each)
        const uint32_t i32 = static_cast<uint32_t>(i), q = i32 / static_cast<uint32_t>(ow);
        const uint32_t im = q / static_cast<uint32_t>(oh);
        ox = static_cast<int>(i32 - q * static_cast<uint32_t>(ow));
        oy = static_cast<int>(q - im * static_cast<uint32_t>(oh));
        img = im;
      } else {
        const long long q = i / ow;
        ox = static_cast<int>(i - q * ow);
        img = q / oh;
        oy = static_cast<int>(q - img * oh);
      }
      const int iy = oy + kh - pad;
      if (iy >= 0 && iy < ih) {
        const float* zr = z + ((img * ih + iy) * iw) * 16 + kh * 4;
        float v[4];
#pragma unroll
        for (int kw = 0; kw < 4; ++kw) {
          const int ix = ox + kw - pad;
          v[kw] = (ix >= 0 && ix < iw) ? __ldg(zr + static_cast<long long>(ix) * 16 + kw) : 0.f;
        }
        s = (v[0] + v[1]) + (v[2] + v[3]);
      }
    }
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    if (kh == 0 && i < total) logits[i] = s + (bias ? __ldg(bias) : 0.f);
  }
}

// u[pix][tap] = dlogits[n][y - kh + pad][x - kw + pad] (zero outside): the column of output gradients
// that input pixel (n, y, x) sees through tap (kh, kw).
__device__ __forceinline__ float gather_dlogit(const float* __restrict__ dlog, long long pix, long long npix, int tap,
                                               int ih, int iw, int oh, int ow, int pad) {
  if (pix >= npix) return 0.f;
  const int x = static_cast<int>(pix % iw);
  const int y = static_cast<int>((pix / iw) % ih);
  const long long img = pix / (static_cast<long long>(iw) * ih);
  const int oy = y - (tap >> 2) + pad, ox = x - (tap & 3) + pad;
  if (oy < 0 || oy >= oh || ox < 0 || ox >= ow) return 0.f;
  return __ldg(dlog + (img * oh + oy) * ow + ox);
}

// Streaming unit of the Cout = 1 kernels: [16 pixels x 64 channels] bf16 = 2 KiB, one full 128-byte line per pixel,
// copied by ONE warp with cp.async into its private ring; the 16-byte granules of a row are XOR-swizzled by (row & 7)
// so that ldmatrix (plain and .trans) and per-lane 128-bit reads of the unit are bank-conflict-free.
constexpr int kC1Ring = 8;     // ring depth of the forward / wgrad kernels (14 KiB in flight per warp)
constexpr int kC1YRing = 4;    // ring depth of the y stream of the backward-fused dgrad (two CTAs per SM)
constexpr int kC1Unit = 2048;
constexpr int kC1Round = 32;   // wgrad: slabs whose gathered dlogits table is built at once (24 KiB)

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, int src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}

// Per-lane invariants of the unit copy (lane -> rows (lane >> 3) + 4 i, granule lane & 7): the first version
// recomputed the 64-bit source addresses and the swizzle per row and unit, ~110 instructions per unit next to the
// ~160 of the MMA loop it feeds (ncu source page of cout1_z2_kernel).
struct C1Lane {
  long long src_off;    // (lane >> 3) * ld + (lane & 7) * 8   (elements)
  long long row_step;   // 4 * ld
  uint32_t dst_off[4];  // swizzled byte offsets of the lane's four granules inside a unit
  int r0;               // lane >> 3
};
__device__ __forceinline__ C1Lane c1_lane(long long ld, uint32_t lane) {
  C1Lane L;
  const uint32_t gran = lane & 7;
  L.r0 = static_cast<int>(lane >> 3);
  L.src_off = L.r0 * ld + gran * 8;
  L.row_step = 4 * ld;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const uint32_t r = (lane >> 3) + 4 * i;
    L.dst_off[i] = r * 128 + ((gran ^ (r & 7)) << 4);
  }
  return L;
}
// one unit: pixels pix0 .. pix0+15 (rows at or beyond pix_end are zero-filled: src-size 0, nothing is read, and the
// address handed to the copy is the tensor's base so that it is a mapped one whatever follows the tensor),
// 64 channels starting at x_ch = x + ch0
__device__ __forceinline__ void c1_issue_unit(uint32_t dst, const bf16* __restrict__ x_ch, long long ld, const C1Lane& L,
                                              long long pix0, long long pix_end) {
  const bf16* src = x_ch + pix0 * ld + L.src_off;
  const long long lim = pix_end - pix0 - L.r0;      // row i of this lane is real iff 4 i < lim
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const bool ok = 4 * i < lim;
    cp_async16(dst + L.dst_off[i], ok ? src + i * L.row_step : x_ch, ok ? 16 : 0);
  }
}

// ------------------------------------------------------------------------------------------------
// Cout = 1 dgrad: gx[pix][c] = sum_tap u[pix][tap] * w[tap][c]   (one k16 MMA step per output tile)
// CTA = 128 input pixels; warp = one 64-channel range, its 8 B fragments held in registers.
// dynamic smem: wT[c][24] | us[128][24] | out_s[8][16][72]   (bf16) | BWD: yring[8 warps][kC1YRing][2 KiB]
// ------------------------------------------------------------------------------------------------
// BWD: the copy-out also applies the activation backward of the layer below (d = (y*scale+shift > 0) ? g : slope*g,
// the LeakyReLU after BatchNorm, models.py:239-240) and accumulates that layer's BatchNorm-backward sums
// [sum d | sum d*y] (of the stored bf16 d) -- the same contract as the tcgen05 dgrad epilogue, so the separate
// reduce pass over y and g disappears.  Needs c <= 512 (one 64-channel range per warp).  The y slabs stream through a
// per-warp cp.async ring (issued kC1YRing - 1 slabs ahead, the first ones before the weight staging): loading them
// with plain global loads right before their use left the kernel bound by that latency (54 us vs 21 us plain).
struct Cout1Bwd {
  const bf16* y;
  long long ld_y;
  const float* scale;
  const float* shift;
  float slope;
  double* sums;
};

template <bool BWD>
__global__ void __launch_bounds__(256, 2) cout1_dgrad_kernel(const float* __restrict__ dlog, int ih, int iw, int oh, int ow,
                                                          int pad, long long npix, const bf16* __restrict__ w, int c,
                                                          bf16* __restrict__ gx, long long ld_gx, const Cout1Bwd b) {
  extern __shared__ __align__(16) uint8_t dsm[];
  bf16* wT = reinterpret_cast<bf16*>(dsm);
  bf16* us = wT + static_cast<size_t>(c) * 24;
  bf16* out_s = us + 128 * 24;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  // BWD: producer / consumer state of this warp's y stream (units in (tile, 16-pixel slab) order)
  const uint8_t* yring = nullptr;
  uint32_t yring_a = 0;
  const C1Lane ylane = c1_lane(BWD ? b.ld_y : 0, static_cast<uint32_t>(lane));
  long long p_tile = blockIdx.x;
  int p_mt = 0, p_unit = 0, c_unit = 0;
  auto y_issue = [&]() {
    if (p_tile * 128 < npix) {
      c1_issue_unit(yring_a + (p_unit & (kC1YRing - 1)) * kC1Unit, b.y + warp * 64, b.ld_y, ylane, p_tile * 128 + p_mt * 16,
                    npix);
      ++p_unit;
      if (++p_mt == 8) {
        p_mt = 0;
        p_tile += gridDim.x;
      }
    }
    cp_async_commit();
  };
  if (BWD && warp * 64 < c) {
    const uint32_t raw = smem_u32(out_s + 8 * 16 * 72);
    const uint32_t al = (raw + 127u) & ~127u;
    yring_a = al + warp * (kC1YRing * kC1Unit);
    yring = reinterpret_cast<const uint8_t*>(out_s + 8 * 16 * 72) + (al - raw) + warp * (kC1YRing * kC1Unit);
#pragma unroll 1
    for (int j = 0; j < kC1YRing - 1; ++j) y_issue();
  }
  {
    // wT[channel][tap] <- w[tap][channel]: 128-bit loads, four per thread issued together, lanes walk the taps so that
    // the 2-byte transposing stores of a half-warp fall into 32 contiguous bytes.  (As one 2-byte load + store per
    // element -- 32 dependent global round trips per thread -- this staging held 33 % / 48 % of the stall samples of
    // the fused / plain kernel: every CTA pays it for only ~1.6 tiles.)
    const int cv = c >> 3, nvec = 16 * cv;
    for (int base = 0; base < nvec; base += 1024) {
      uint4 q[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int k = base + tid + i * 256, tap = k & 15, seg = k >> 4;
        q[i] = k < nvec ? ldg128(w + static_cast<long long>(tap) * c + seg * 8) : make_uint4(0, 0, 0, 0);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int k = base + tid + i * 256, tap = k & 15, seg = k >> 4;
        if (k < nvec) {
          const uint32_t wd[4] = {q[i].x, q[i].y, q[i].z, q[i].w};
          unsigned short* d = reinterpret_cast<unsigned short*>(wT) + seg * 8 * 24 + tap;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            d[(2 * j) * 24] = static_cast<unsigned short>(wd[j] & 0xffffu);
            d[(2 * j + 1) * 24] = static_cast<unsigned short>(wd[j] >> 16);
          }
        }
      }
    }
  }
  const uint32_t us_a = smem_u32(us);
  bf16* my_out = out_s + warp * 16 * 72;
  // BWD: this lane always copies out the same 8 channels (warp's 64-channel range, segment lane & 7)
  float bsc[8], bsh[8], s1[8], s2[8];
  if (BWD) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int ch = warp * 64 + (lane & 7) * 8 + j;
      bsc[j] = ch < c ? __ldg(b.scale + ch) : 0.f;
      bsh[j] = ch < c ? __ldg(b.shift + ch) : 0.f;
      s1[j] = s2[j] = 0.f;
    }
  }
  for (long long tile = blockIdx.x; tile * 128 < npix; tile += gridDim.x) {
    __syncthreads();  // wT ready (first pass) / previous tile's us consumed
    {
      // one pixel and eight taps (two kernel rows) per thread: ONE (n, y, x) decomposition instead of eight 64-bit ones
      // (the staging, not the stores, bounded this kernel), one 128-bit shared-memory store
      const int px = tid & 127, kh0 = (tid >> 7) * 2;
      const long long pix = tile * 128 + px;
      uint32_t pk[4] = {0u, 0u, 0u, 0u};
      if (pix < npix) {
        int xx, yy;
        long long img;
        if (npix <= 0x7fffffffLL) {
          const uint32_t p32 = static_cast<uint32_t>(pix), q = p32 / static_cast<uint32_t>(iw);
          xx = static_cast<int>(p32 - q * static_cast<uint32_t>(iw));
          const uint32_t im = q / static_cast<uint32_t>(ih);
          yy = static_cast<int>(q - im * static_cast<uint32_t>(ih));
          img = im;
        } else {
          xx = static_cast<int>(pix % iw);
          yy = static_cast<int>((pix / iw) % ih);
          img = pix / (static_cast<long long>(iw) * ih);
        }
        const float* dl = dlog + img * oh * ow;
#pragma unroll
        for (int j2 = 0; j2 < 4; ++j2) {
          float v[2];
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int j = 2 * j2 + e;
            const int oy = yy - (kh0 + (j >> 2)) + pad, ox = xx - (j & 3) + pad;
            v[e] = (oy >= 0 && oy < oh && ox >= 0 && ox < ow) ? __ldg(dl + oy * ow + ox) : 0.f;
          }
          pk[j2] = pack_bf16x2(v[0], v[1]);
        }
      }
      *reinterpret_cast<uint4*>(us + px * 24 + kh0 * 4) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    }
    __syncthreads();
    for (int nr = warp; nr < (c >> 6); nr += 8) {
      const int n0 = nr * 64;
      uint32_t bfr[8][2];
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        const bf16* row = wT + (n0 + nt * 8 + g) * 24;
        bfr[nt][0] = *reinterpret_cast<const uint32_t*>(row + 2 * t);
        bfr[nt][1] = *reinterpret_cast<const uint32_t*>(row + 2 * t + 8);
      }
      for (int mt = 0; mt < 8; ++mt) {
        const uint8_t* ystage = nullptr;
        if (BWD) {
          cp_async_wait<kC1YRing - 2>();
          __syncwarp();          // this slab's y rows have landed for every lane; the previous slab's reads are done
          y_issue();             // refills the stage read one iteration ago
          ystage = yring + (c_unit & (kC1YRing - 1)) * kC1Unit;
          ++c_unit;
        }
        uint32_t a[4];
        lda_16x16(a, us_a + mt * 16 * 48, 48, lane);
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          float acc[4] = {0.f, 0.f, 0.f, 0.f};
          mma_bf16_16816(acc, a, bfr[nt][0], bfr[nt][1]);
          *reinterpret_cast<uint32_t*>(my_out + g * 72 + nt * 8 + 2 * t) = pack_bf16x2(acc[0], acc[1]);
          *reinterpret_cast<uint32_t*>(my_out + (g + 8) * 72 + nt * 8 + 2 * t) = pack_bf16x2(acc[2], acc[3]);
        }
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int idx = lane + i * 32, r = idx >> 3, seg = idx & 7;
          const long long pix = tile * 128 + mt * 16 + r;
          if (pix < npix) {
            uint4 v = *reinterpret_cast<const uint4*>(my_out + r * 72 + seg * 8);
            if (BWD) {
              const uint4 yv = *reinterpret_cast<const uint4*>(ystage + r * 128 + ((seg ^ (r & 7)) << 4));
              const uint32_t gw[4] = {v.x, v.y, v.z, v.w}, yw[4] = {yv.x, yv.y, yv.z, yv.w};
              uint32_t pk[4];
#pragma unroll
              for (int j2 = 0; j2 < 4; ++j2) {
                float d[2];
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                  const int j = 2 * j2 + e;
                  const float gj = e ? bf16_hi(gw[j2]) : bf16_lo(gw[j2]);
                  const float yj = e ? bf16_hi(yw[j2]) : bf16_lo(yw[j2]);
                  d[e] = fmaf(yj, bsc[j], bsh[j]) > 0.f ? gj : b.slope * gj;
                }
                pk[j2] = pack_bf16x2(d[0], d[1]);
#pragma unroll
                for (int e = 0; e < 2; ++e) {      // sums of the stored (bf16-rounded) values
                  const int j = 2 * j2 + e;
                  const float dj = e ? bf16_hi(pk[j2]) : bf16_lo(pk[j2]);
                  const float yj = e ? bf16_hi(yw[j2]) : bf16_lo(yw[j2]);
                  s1[j] += dj;
                  s2[j] = fmaf(dj, yj, s2[j]);
                }
              }
              v = make_uint4(pk[0], pk[1], pk[2], pk[3]);
            }
            *reinterpret_cast<uint4*>(gx + pix * ld_gx + n0 + seg * 8) = v;
          }
        }
        __syncwarp();
      }
    }
  }
  if (BWD) {
    cp_async_wait<0>();
    // lanes l, l+8, l+16, l+24 hold the same channels
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      s1[j] += __shfl_xor_sync(0xffffffffu, s1[j], 8);
      s1[j] += __shfl_xor_sync(0xffffffffu, s1[j], 16);
      s2[j] += __shfl_xor_sync(0xffffffffu, s2[j], 8);
      s2[j] += __shfl_xor_sync(0xffffffffu, s2[j], 16);
    }
    if (lane < 8 && warp * 64 < c) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int ch = warp * 64 + lane * 8 + j;
        atomicAdd(b.sums + ch, static_cast<double>(s1[j]));
        atomicAdd(b.sums + c + ch, static_cast<double>(s2[j]));
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Cout = 1 wgrad: dw[tap][c] += sum_pix u[pix][tap] * x[pix][c]   (K = pixels)
// CTA = a contiguous range of input pixels; warp = one 64-channel range (c <= 512).
// dynamic smem: xs[16][c + 8] | ut[16][24]   (bf16)
// ------------------------------------------------------------------------------------------------
// PRE: x = LeakyReLU(y*scale + shift) is formed from the raw conv output y while staging (see cout1_z_kernel).
// The next 16-pixel slab's global loads are in flight while the current slab's MMAs run (register prefetch;
// kVec = uint4 per thread and slab = 16 * c / 8 / 256, i.e. 4 for c = 512).
template <bool PRE>
__global__ void __launch_bounds__(256, 4) cout1_wgrad_kernel(const float* __restrict__ dlog, int ih, int iw, int oh, int ow,
                                                          int pad, long long npix, long long chunk,
                                                          const bf16* __restrict__ x, long long ld_x, int c,
                                                          float* __restrict__ dw, const Cout1Pre pre) {
  extern __shared__ __align__(16) uint8_t dsm[];
  bf16* xs = reinterpret_cast<bf16*>(dsm);
  const int xstride = c + 8;
  bf16* ut = xs + 16 * xstride;
  float* par = reinterpret_cast<float*>(ut + 16 * 24);   // scale[c] | shift[c] (PRE only)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const long long p0 = blockIdx.x * chunk, p1 = min(npix, p0 + chunk);
  const uint32_t xs_a = smem_u32(xs), ut_a = smem_u32(ut);
  const int n0 = warp * 64;
  const bool active = n0 < c;
  float acc[8][4];
#pragma unroll
  for (int nt = 0; nt < 8; ++nt)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[nt][j] = 0.f;
  const int vec_per_px = c >> 3;
  const int n_vec = 16 * vec_per_px;        // <= 1024 (c <= 512): at most 4 per thread
  // vec_per_px (c / 8) divides 256 for the supported c in {64, 128, 256, 512}: idx % vec_per_px = tid % vec_per_px for
  // every i, so a thread always stages the same 8 channels; their scale / shift sit in shared memory as one 32-byte row
  // per channel group (two 128-bit loads per slab: registers are needed for the 32 accumulators and the prefetch)
  if (PRE) {
    for (int i = tid; i < c; i += 256) {
      par[i] = __ldg(pre.scale + i);
      par[c + i] = __ldg(pre.shift + i);
    }
    __syncthreads();
  }
  const int my_ch = (tid % vec_per_px) * 8;
  uint4 nxt[4];
  float unxt = 0.f;
  auto fetch = [&](long long k0) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = tid + i * 256;
      nxt[i] = make_uint4(0, 0, 0, 0);
      if (idx < n_vec) {
        const int px = idx / vec_per_px, seg = idx - px * vec_per_px;
        const long long pix = k0 + px;
        if (pix < p1) nxt[i] = ldg128(x + pix * ld_x + seg * 8);
      }
    }
    const int tap = tid >> 4, px = tid & 15;
    const long long pix = k0 + px;
    unxt = pix < p1 ? gather_dlogit(dlog, pix, npix, tap, ih, iw, oh, ow, pad) : 0.f;
  };
  if (p0 < p1) fetch(p0);
  for (long long k0 = p0; k0 < p1; k0 += 16) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = tid + i * 256;
      if (idx < n_vec) {
        const int px = idx / vec_per_px, seg = idx - px * vec_per_px;
        uint4 val = nxt[i];
        if (PRE && k0 + px < p1) {
          float sc[8], sh[8];
          lds8(par + my_ch, sc);
          lds8(par + c + my_ch, sh);
          val = bn_act8(val, sc, sh, pre.slope);
        }
        *reinterpret_cast<uint4*>(xs + px * xstride + seg * 8) = val;
      }
    }
    ut[(tid >> 4) * 24 + (tid & 15)] = __float2bfloat16(unxt);
    __syncthreads();
    if (k0 + 16 < p1) fetch(k0 + 16);
    if (active) {
      uint32_t a[4];
      lda_16x16(a, ut_a, 48, lane);
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        uint32_t b0, b1;
        ldmatrix_x2_trans(b0, b1, xs_a + ((lane & 15) * xstride + n0 + nt * 8) * 2);
        mma_bf16_16816(acc[nt], a, b0, b1);
      }
    }
    __syncthreads();
  }
  if (active && p1 > p0) {       // (warp-uniform: the shuffles below are executed by whole warps)
    // One 128-bit reduction per lane and 8-column block instead of four scalar ones (every CTA adds its whole
    // 16 x c partial to the same 16 x c words: the L2 atomic units, not the loads, bounded this kernel): lanes t and
    // t ^ 1 swap halves so that the even lane owns 4 consecutive columns of tap row g, the odd lane those of row g + 8.
    const bool odd = t & 1;
    const bool vec = (reinterpret_cast<uintptr_t>(dw) & 15) == 0;      // c % 64 == 0 keeps every row 16-byte aligned
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const float s0 = odd ? acc[nt][0] : acc[nt][2], s1 = odd ? acc[nt][1] : acc[nt][3];
      const float r0 = __shfl_xor_sync(0xffffffffu, s0, 1), r1 = __shfl_xor_sync(0xffffffffu, s1, 1);
      const int col = n0 + nt * 8 + 4 * (t >> 1);
      float* dst = dw + static_cast<long long>(odd ? g + 8 : g) * c + col;
      const float v0 = odd ? r0 : acc[nt][0], v1 = odd ? r1 : acc[nt][1];
      const float v2 = odd ? acc[nt][2] : r0, v3 = odd ? acc[nt][3] : r1;
      if (vec) {
        red_add_v4_f32(dst, v0, v1, v2, v3);
      } else {
        atomicAdd(dst, v0);
        atomicAdd(dst + 1, v1);
        atomicAdd(dst + 2, v2);
        atomicAdd(dst + 3, v3);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Streaming versions of the Cout = 1 forward and weight gradient (c <= 512, 0 <= slope <= 1, < 2^31 pixels; the
// kernels above stay as the general path).  The kernels above hold ONE 16 KiB chunk per CTA in flight between two
// __syncthreads (1.4-1.9 TB/s on the 63 MB head input).  Here every warp streams its own [16 pixels x 64 channels]
// units (2 KiB: one full 128-byte line per pixel) through a private ring of eight cp.async stages, so a CTA of
// eight warps keeps 112 KiB in flight without any CTA-wide barrier in the load path; the 16-byte granules of a
// row are XOR-swizzled by (row & 7), which makes both ldmatrix forms below conflict-free.  BatchNorm + LeakyReLU of
// the layer below (PRE) are applied to the MMA FRAGMENTS (a lane always sees the same channels, so its scale /
// shift sit in registers); LeakyReLU is max(v, slope*v).
// ------------------------------------------------------------------------------------------------
// two packed bf16 values -> LeakyReLU(v*scale + shift) with one (scale, shift) pair per half
__device__ __forceinline__ uint32_t bn_lrelu2(uint32_t v, float sc_lo, float sh_lo, float sc_hi, float sh_hi, float slope) {
  const float a = fmaf(bf16_lo(v), sc_lo, sh_lo), b = fmaf(bf16_hi(v), sc_hi, sh_hi);
  return pack_bf16x2(fmaxf(a, slope * a), fmaxf(b, slope * b));
}

// Forward stage 1 (z[pix][tap], as cout1_z_kernel).  CTA tile = 32 pixels: warp = (16-pixel slab, quarter of the
// channels); its B fragments (the weights of its <= 2 chunks) and PRE parameters stay in registers for the whole
// kernel.  The four K quarters of a slab are summed through shared memory (double-buffered: one barrier per tile).
// dynamic smem: ring[8 warps][kC1Ring][2 KiB] | red[2][8][256] fp32
template <bool PRE>
__global__ void __launch_bounds__(256, 1) cout1_z2_kernel(const bf16* __restrict__ x, long long ld_x, int npix, int c,
                                                          const bf16* __restrict__ w, float* __restrict__ z,
                                                          const Cout1Pre pre) {
  extern __shared__ __align__(16) uint8_t dsm[];
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const uint32_t sbase = (smem_u32(dsm) + 127u) & ~127u;      // 128-byte rows: the swizzle assumes aligned units
  const uint32_t ring = sbase + warp * (kC1Ring * kC1Unit);
  float* red = reinterpret_cast<float*>(dsm + (sbase - smem_u32(dsm)) + 8 * kC1Ring * kC1Unit);
  const int sj = warp >> 2, kq = warp & 3;
  const int nch = c >> 6;
  const int cpw = (nch + 3) >> 2;                                  // chunks per warp (<= 2)
  const int ch_first = kq * cpw;
  const int my_chunks = max(0, min(cpw, nch - ch_first));
  const int ntiles = (npix + 31) >> 5;
  const int my_tiles = static_cast<int>(blockIdx.x) < ntiles ? (ntiles - 1 - static_cast<int>(blockIdx.x)) / static_cast<int>(gridDim.x) + 1 : 0;
  const int n_units = my_tiles * my_chunks;

  // producer state: unit -> (tile, chunk)
  const C1Lane xlane = c1_lane(ld_x, lane);
  int p_unit = 0, p_ti = 0, p_cc = 0;
  auto issue_next = [&]() {
    if (p_unit < n_units) {
      const long long pix0 = (static_cast<long long>(blockIdx.x) + static_cast<long long>(p_ti) * gridDim.x) * 32 + sj * 16;
      c1_issue_unit(ring + (p_unit & (kC1Ring - 1)) * kC1Unit, x + (ch_first + p_cc) * 64, ld_x, xlane, pix0, npix);
      ++p_unit;
      if (++p_cc == my_chunks) {
        p_cc = 0;
        ++p_ti;
      }
    }
    cp_async_commit();
  };
#pragma unroll 1
  for (int j = 0; j < kC1Ring - 1; ++j) issue_next();

  uint32_t bq[2][4][4];      // [chunk][k step]{n tile 0: b0 b1 | n tile 1: b0 b1}
  float sc[2][4][4], sh[2][4][4];
#pragma unroll
  for (int cc = 0; cc < 2; ++cc) {
    const bool have = cc < my_chunks;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const int cb = (ch_first + cc) * 64 + ks * 16 + 2 * t;
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        const bf16* wr = w + static_cast<long long>(nt * 8 + g) * c + cb;
        bq[cc][ks][2 * nt] = have ? __ldg(reinterpret_cast<const uint32_t*>(wr)) : 0u;
        bq[cc][ks][2 * nt + 1] = have ? __ldg(reinterpret_cast<const uint32_t*>(wr + 8)) : 0u;
      }
      if (PRE) {
        const int off[4] = {0, 1, 8, 9};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          sc[cc][ks][j] = have ? __ldg(pre.scale + cb + off[j]) : 0.f;
          sh[cc][ks][j] = have ? __ldg(pre.shift + cb + off[j]) : 0.f;
        }
      }
    }
  }

  int stage = 0;
  for (int ti = 0; ti < my_tiles; ++ti) {
    float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
    for (int cc = 0; cc < 2; ++cc) {
      if (cc < my_chunks) {
        cp_async_wait<kC1Ring - 2>();
        __syncwarp();            // every lane's copies of this unit have landed; the previous unit's reads are done
        issue_next();            // refills the stage consumed one iteration ago
        const uint32_t ub = ring + stage * kC1Unit;
        stage = (stage + 1) & (kC1Ring - 1);
        const uint32_t r = lane & 15;
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          uint32_t a[4];
          ldmatrix_x4(a, ub + r * 128 + (((2 * ks + (lane >> 4)) ^ (r & 7)) << 4));
          if (PRE) {
            a[0] = bn_lrelu2(a[0], sc[cc][ks][0], sh[cc][ks][0], sc[cc][ks][1], sh[cc][ks][1], pre.slope);
            a[1] = bn_lrelu2(a[1], sc[cc][ks][0], sh[cc][ks][0], sc[cc][ks][1], sh[cc][ks][1], pre.slope);
            a[2] = bn_lrelu2(a[2], sc[cc][ks][2], sh[cc][ks][2], sc[cc][ks][3], sh[cc][ks][3], pre.slope);
            a[3] = bn_lrelu2(a[3], sc[cc][ks][2], sh[cc][ks][2], sc[cc][ks][3], sh[cc][ks][3], pre.slope);
          }
          mma_bf16_16816(acc[0], a, bq[cc][ks][0], bq[cc][ks][1]);
          mma_bf16_16816(acc[1], a, bq[cc][ks][2], bq[cc][ks][3]);
        }
      }
    }
    float* rb = red + ((ti & 1) * 8 + warp) * 256;
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) {
      *reinterpret_cast<float2*>(rb + g * 16 + nt * 8 + 2 * t) = make_float2(acc[nt][0], acc[nt][1]);
      *reinterpret_cast<float2*>(rb + (g + 8) * 16 + nt * 8 + 2 * t) = make_float2(acc[nt][2], acc[nt][3]);
    }
    __syncthreads();
    // thread -> two consecutive taps of one pixel: sum of the four K quarters of its slab
    const int o = tid * 2, oj = o >> 8, idx = o & 255;
    const float* rs = red + ((ti & 1) * 8 + oj * 4) * 256 + idx;
    float2 s = *reinterpret_cast<const float2*>(rs);
#pragma unroll
    for (int q = 1; q < 4; ++q) {
      const float2 v = *reinterpret_cast<const float2*>(rs + q * 256);
      s.x += v.x;
      s.y += v.y;
    }
    const long long pix = (static_cast<long long>(blockIdx.x) + static_cast<long long>(ti) * gridDim.x) * 32 + oj * 16 + (idx >> 4);
    if (pix < npix) *reinterpret_cast<float2*>(z + pix * 16 + (idx & 15)) = s;
  }
  cp_async_wait<0>();
}

// Weight gradient (as cout1_wgrad_kernel): CTA = a contiguous pixel range, warp = one 64-channel range with its
// 16 x 64 accumulator in registers over the whole range; the gathered output gradients u[tap][pixel] of up to
// kC1Round slabs are tabulated in shared memory by the whole CTA (one (n, y, x) decomposition per pixel, 32-bit)
// while the first units are already in flight.  One CTA per SM: 148 partial flushes instead of 592.
// dynamic smem: ring[8 warps][kC1Ring][2 KiB] | U[kC1Round][16 taps][24] bf16
template <bool PRE>
__global__ void __launch_bounds__(256, 1) cout1_wgrad2_kernel(const float* __restrict__ dlog, int ih, int iw, int oh, int ow,
                                                              int pad, int npix, int chunk, const bf16* __restrict__ x,
                                                              long long ld_x, int c, float* __restrict__ dw,
                                                              const Cout1Pre pre) {
  extern __shared__ __align__(16) uint8_t dsm[];
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const uint32_t sbase = (smem_u32(dsm) + 127u) & ~127u;
  const uint32_t ring = sbase + warp * (kC1Ring * kC1Unit);
  bf16* U = reinterpret_cast<bf16*>(dsm + (sbase - smem_u32(dsm)) + 8 * kC1Ring * kC1Unit);
  const uint32_t U_a = smem_u32(U);
  const int p0 = static_cast<int>(blockIdx.x) * chunk, p1 = min(npix, p0 + chunk);
  const int n_slabs = (p1 - p0 + 15) >> 4;
  const int n0 = warp * 64;
  const bool active = n0 < c;
  const C1Lane xlane = c1_lane(ld_x, lane);
  int p_slab = 0;
  auto issue_next = [&]() {
    if (p_slab < n_slabs) {
      c1_issue_unit(ring + (p_slab & (kC1Ring - 1)) * kC1Unit, x + n0, ld_x, xlane, p0 + 16 * p_slab, p1);
      ++p_slab;
    }
    cp_async_commit();
  };
  if (active) {
#pragma unroll 1
    for (int j = 0; j < kC1Ring - 1; ++j) issue_next();
  }
  float sc[8], sh[8];
  if (PRE) {
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      sc[nt] = active ? __ldg(pre.scale + n0 + nt * 8 + g) : 0.f;
      sh[nt] = active ? __ldg(pre.shift + n0 + nt * 8 + g) : 0.f;
    }
  }
  float acc[8][4];
#pragma unroll
  for (int nt = 0; nt < 8; ++nt)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[nt][j] = 0.f;

  for (int r0 = 0; r0 < n_slabs; r0 += kC1Round) {
    const int rs = min(kC1Round, n_slabs - r0);
    if (r0) __syncthreads();        // the previous round's table has been consumed
    for (int i = tid; i < rs * 16; i += 256) {
      const int pix = p0 + r0 * 16 + i;
      bf16* ur = U + (i >> 4) * (16 * 24) + (i & 15);
      if (pix < p1) {
        const int xx = pix % iw, q = pix / iw, yy = q % ih, img = q / ih;
        const float* dl = dlog + static_cast<long long>(img) * oh * ow;
#pragma unroll
        for (int tap = 0; tap < 16; ++tap) {
          const int oy = yy - (tap >> 2) + pad, ox = xx - (tap & 3) + pad;
          const bool in = oy >= 0 && oy < oh && ox >= 0 && ox < ow;
          ur[tap * 24] = __float2bfloat16(in ? __ldg(dl + oy * ow + ox) : 0.f);
        }
      } else {
#pragma unroll
        for (int tap = 0; tap < 16; ++tap) ur[tap * 24] = __float2bfloat16(0.f);
      }
    }
    __syncthreads();
    if (active) {
      for (int s = 0; s < rs; ++s) {
        cp_async_wait<kC1Ring - 2>();
        __syncwarp();
        issue_next();
        const uint32_t ub = ring + ((r0 + s) & (kC1Ring - 1)) * kC1Unit;
        uint32_t a[4];
        lda_16x16(a, U_a + s * (16 * 48), 48, lane);
        const uint32_t r = lane & 15;
#pragma unroll
        for (int np = 0; np < 4; ++np) {
          uint32_t b[4];
          ldmatrix_x4_trans(b, ub + r * 128 + (((2 * np + (lane >> 4)) ^ (r & 7)) << 4));
          if (PRE) {
            b[0] = bn_lrelu2(b[0], sc[2 * np], sh[2 * np], sc[2 * np], sh[2 * np], pre.slope);
            b[1] = bn_lrelu2(b[1], sc[2 * np], sh[2 * np], sc[2 * np], sh[2 * np], pre.slope);
            b[2] = bn_lrelu2(b[2], sc[2 * np + 1], sh[2 * np + 1], sc[2 * np + 1], sh[2 * np + 1], pre.slope);
            b[3] = bn_lrelu2(b[3], sc[2 * np + 1], sh[2 * np + 1], sc[2 * np + 1], sh[2 * np + 1], pre.slope);
          }
          mma_bf16_16816(acc[2 * np], a, b[0], b[1]);
          mma_bf16_16816(acc[2 * np + 1], a, b[2], b[3]);
        }
      }
    }
  }
  cp_async_wait<0>();
  if (active && p1 > p0) {       // same flush as cout1_wgrad_kernel: one 128-bit reduction per lane and 8-column block
    const bool odd = t & 1;
    const bool vec = (reinterpret_cast<uintptr_t>(dw) & 15) == 0;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      const float s0 = odd ? acc[nt][0] : acc[nt][2], s1 = odd ? acc[nt][1] : acc[nt][3];
      const float r0 = __shfl_xor_sync(0xffffffffu, s0, 1), r1 = __shfl_xor_sync(0xffffffffu, s1, 1);
      const int col = n0 + nt * 8 + 4 * (t >> 1);
      float* dst = dw + static_cast<long long>(odd ? g + 8 : g) * c + col;
      const float v0 = odd ? r0 : acc[nt][0], v1 = odd ? r1 : acc[nt][1];
      const float v2 = odd ? acc[nt][2] : r0, v3 = odd ? acc[nt][3] : r1;
      if (vec) {
        red_add_v4_f32(dst, v0, v1, v2, v3);
      } else {
        atomicAdd(dst, v0);
        atomicAdd(dst + 1, v1);
        atomicAdd(dst + 2, v2);
        atomicAdd(dst + 3, v3);
      }
    }
  }
}


// ------------------------------------------------------------------------------------------------
// Thin-input Conv2d(k4, s2, p1): out[pix][cw] = sum_{tap, slot} in[2*pix + tap - 1][slot] * w[cw][tap][slot]
// for inputs of 3 channels (one NHWC source with 4 channel slots, CT = 4) or 6 channels (two such
// sources concatenated, CT = 8): the generator's first conv (models.py:177 outermost), the
// discriminator's first conv on cat(A, B) (models.py:223, train_gan.py:57) and the input gradient of the
// generator's last ConvTranspose2d (models.py:184).  The input patch of an 8 x 16 output tile is staged in
// shared memory once and the im2col matrix only ever exists as MMA fragments.
// CTA = 128 output pixels; warp = 2 output rows (2 x m16) x 64 output channels.
// The output tile leaves through TMA stores from a 128B-swizzled smem tile (ragged tiles are clipped by the unit):
// the per-thread copy-out loop it replaces was ~19 % of the kernel's instructions (ncu source page).
// dynamic smem (1 KiB aligned): out_s[cw/64][128][128 B] | patch[2][18][34][CT] (cp.async double buffer) | ws[cw][16*CT + 8]
// ------------------------------------------------------------------------------------------------
struct ThinFwdParams {
  CUtensorMap tm_out[2];   // out1 / out2 as [n][oh][ow][cw] bf16: box 64 ch x 16 x 8 x 1, 128B swizzle (TMA store)
  CUtensorMap tm_row[2];   // the same tensors, box 64 ch x 128 x 1 x 1: one output row (tcgen05 row kernel)
  const bf16* s0;
  long long ld0;
  const bf16* s1;
  long long ld1;
  const bf16* w;
  const float* bias;
  int n, h, w_in, oh, ow, cw;
  bf16* out1;
  long long ldo1;
  float slope1;
  bf16* out2;
  long long ldo2;
  float slope2;
  int tiles_x, tiles_y;
  long long total_tiles;
  int skip;  // bring-up ablation: 1 no MMA loop, 2 no global stores, 4 no patch loads
};

template <int CT>
__global__ void __launch_bounds__(256) thin_conv_fwd_kernel(const __grid_constant__ ThinFwdParams p) {
  constexpr int K = 16 * CT;
  constexpr int WSTRIDE = K + 8;      // bf16 elements per weight row in smem
  constexpr int PW = CT / 2;          // 32-bit words per patch pixel
  extern __shared__ uint8_t dsm_raw[];
  const uint32_t out_a = (smem_u32(dsm_raw) + 1023u) & ~1023u;             // out_s: cw/64 swizzled tiles of 16 KiB
  uint8_t* dsm = dsm_raw + (out_a - smem_u32(dsm_raw));
  constexpr int PATCH_WORDS = 18 * 34 * PW;
  const int out_bytes = (p.cw >> 6) * 16384;
  uint32_t* patch_buf = reinterpret_cast<uint32_t*>(dsm + out_bytes);      // [2][18][34][PW]
  bf16* ws = reinterpret_cast<bf16*>(dsm + out_bytes + 2 * PATCH_WORDS * 4);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int mp = warp & 3, nh = warp >> 2;
  const int nthr = blockDim.x;

  for (int idx = tid; idx < p.cw * (K / 8); idx += nthr) {
    const int r = idx / (K / 8), seg = idx - r * (K / 8);
    *reinterpret_cast<uint4*>(ws + r * WSTRIDE + seg * 8) = ldg128(p.w + static_cast<long long>(r) * K + seg * 8);
  }
  const uint32_t ws_a = smem_u32(ws);

  // asynchronous (cp.async) load of the input patch of one tile into a patch buffer
  auto issue_patch = [&](long long tile, int buf) {
    const int t32 = static_cast<int>(tile), tpi = p.tiles_x * p.tiles_y;   // 32-bit: 64-bit division is ~10 % of the kernel
    const int img32 = t32 / tpi, rem32 = t32 - img32 * tpi;
    const int ty = rem32 / p.tiles_x, tx = rem32 - ty * p.tiles_x;
    const long long img = img32;
    const int oy0 = ty * 8, ox0 = tx * 16;
    const bf16* s0i = p.s0 + img * p.h * p.w_in * p.ld0;
    const bf16* s1i = CT == 8 ? p.s1 + img * p.h * p.w_in * p.ld1 : p.s0;
    const int ld0 = static_cast<int>(p.ld0), ld1 = static_cast<int>(p.ld1);
    const uint32_t dst0 = smem_u32(patch_buf + buf * PATCH_WORDS);
    for (int idx = tid; idx < 18 * 34; idx += nthr) {
      const int py = idx / 34, px = idx - py * 34;
      const int iy = 2 * oy0 - 1 + py, ix = 2 * ox0 - 1 + px;
      const bool ok = static_cast<unsigned>(iy) < static_cast<unsigned>(p.h) &&
                      static_cast<unsigned>(ix) < static_cast<unsigned>(p.w_in) && !(p.skip & 4);
      const int pix = ok ? iy * p.w_in + ix : 0;
      cp_async8(dst0 + idx * PW * 4, s0i + pix * ld0, ok ? 8 : 0);
      if (CT == 8) cp_async8(dst0 + idx * PW * 4 + 8, s1i + pix * ld1, ok ? 8 : 0);
    }
    cp_async_commit();
  };

  if (static_cast<long long>(blockIdx.x) < p.total_tiles) issue_patch(blockIdx.x, 0);
  int buf = 0;
  for (long long tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, buf ^= 1) {
    const int t32 = static_cast<int>(tile), tpi = p.tiles_x * p.tiles_y;   // 32-bit: 64-bit division is ~10 % of the kernel
    const int img32 = t32 / tpi, rem32 = t32 - img32 * tpi;
    const int ty = rem32 / p.tiles_x, tx = rem32 - ty * p.tiles_x;
    const long long img = img32;
    const int oy0 = ty * 8, ox0 = tx * 16;
    const uint32_t* patch = patch_buf + buf * PATCH_WORDS;
    const long long next = tile + gridDim.x;
    // the other patch buffer was last read two iterations ago (a __syncthreads lies in between)
    if (next < p.total_tiles) {
      issue_patch(next, buf ^ 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    if (tid == 0) tma_store_wait_read();   // the previous tile's TMA stores have read out_s
    __syncthreads();  // this tile's patch has landed for every thread; out_s of the previous tile is free; ws loaded

    float acc[2][8][4];
#pragma unroll
    for (int m = 0; m < 2; ++m)
#pragma unroll
      for (int nt = 0; nt < 8; ++nt)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[m][nt][j] = 0.f;

    if (!(p.skip & 1))
#pragma unroll
    for (int ks = 0; ks < K / 16; ++ks) {
      uint32_t a[2][4];
#pragma unroll
      for (int m = 0; m < 2; ++m) {
        const int oyl = 2 * mp + m;
        if (CT == 8) {
          const int tap0 = 2 * ks, kh = tap0 >> 2, kw = tap0 & 3;
          const int base = ((2 * oyl + kh) * 34 + kw) * PW + t;
          a[m][0] = patch[base + (2 * g) * PW];
          a[m][1] = patch[base + (2 * (g + 8)) * PW];
          a[m][2] = patch[base + (2 * g + 1) * PW];
          a[m][3] = patch[base + (2 * (g + 8) + 1) * PW];
        } else {
          const int kh = ks, kw = t >> 1;
          const int base = ((2 * oyl + kh) * 34 + kw) * PW + (t & 1);
          a[m][0] = patch[base + (2 * g) * PW];
          a[m][1] = patch[base + (2 * (g + 8)) * PW];
          a[m][2] = patch[base + (2 * g + 2) * PW];
          a[m][3] = patch[base + (2 * (g + 8) + 2) * PW];
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint32_t b[4];
        ldb_16x16(b, ws_a + ((nh * 64 + j * 16) * WSTRIDE + ks * 16) * 2, WSTRIDE * 2, lane);
#pragma unroll
        for (int m = 0; m < 2; ++m) {
          mma_bf16_16816(acc[m][2 * j], a[m], b[0], b[1]);
          mma_bf16_16816(acc[m][2 * j + 1], a[m], b[2], b[3]);
        }
      }
    }

    if (p.bias != nullptr) {
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        const int col = nh * 64 + nt * 8 + 2 * t;
        const float b0 = __ldg(p.bias + col), b1 = __ldg(p.bias + col + 1);
#pragma unroll
        for (int m = 0; m < 2; ++m) {
          acc[m][nt][0] += b0;
          acc[m][nt][1] += b1;
          acc[m][nt][2] += b0;
          acc[m][nt][3] += b1;
        }
      }
    }
    for (int pass = 0; pass < 2; ++pass) {
      bf16* outp = pass == 0 ? p.out1 : p.out2;
      if (outp == nullptr) break;
      const float slope = pass == 0 ? p.slope1 : p.slope2;
      const __nv_bfloat162 slope2 = __float2bfloat162_rn(slope);
      const bool ident = slope == 1.f;
      if (pass == 1) {
        if (tid == 0) tma_store_wait_read();
        __syncthreads();
      }
#pragma unroll
      for (int m = 0; m < 2; ++m) {
        // 128B-swizzled [128 pixels][64 ch] tile per channel half: 16-byte chunk c of row r lives at chunk c ^ (r & 7)
        // (g = r & 7 here, so the eight rows of a warp store hit eight different chunks: conflict-free)
        const int r0 = (2 * mp + m) * 16 + g;
        const uint32_t row0 = out_a + nh * 16384 + r0 * 128 + 4 * t;
        const uint32_t row1 = row0 + 8 * 128;      // row r0 + 8: same r & 7
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          // act(v) = max(v, slope*v) for slope in [0,1], applied to the packed bf16 pair
          __nv_bfloat162 lo = __floats2bfloat162_rn(acc[m][nt][0], acc[m][nt][1]);
          __nv_bfloat162 hi = __floats2bfloat162_rn(acc[m][nt][2], acc[m][nt][3]);
          if (!ident) {
            lo = __hmax2(lo, __hmul2(lo, slope2));
            hi = __hmax2(hi, __hmul2(hi, slope2));
          }
          const uint32_t sw = static_cast<uint32_t>((nt ^ g) << 4);
          st_shared_b32(row0 + sw, *reinterpret_cast<const uint32_t*>(&lo));
          st_shared_b32(row1 + sw, *reinterpret_cast<const uint32_t*>(&hi));
        }
      }
      fence_proxy_async_smem();
      __syncthreads();
      if (tid == 0 && !(p.skip & 2)) {
        for (int b = 0; b < (p.cw >> 6); ++b)
          tma_store_4d(&p.tm_out[pass], out_a + b * 16384, b * 64, ox0, oy0, static_cast<int>(img));
        tma_store_commit();
      }
    }
  }
  if (tid == 0) tma_store_wait_all();
}


// ------------------------------------------------------------------------------------------------
// The same convolution on tcgen05 for full-width rows (w_in = 256, dense 4-slot sources): one output row of 128 pixels
// is one M = 128 accumulator tile, and the im2col matrix is never built -- the A descriptors read it straight out of
// the staged image rows with the un-swizzled K-major layout (ptx.cuh make_nosw_desc), whose 8-row core matrices only
// need rows 16 bytes apart:
//   CT = 8 (two sources, 16 B per concatenated pixel): a row is staged as two planes of 130 entries, odd pixels
//     (entry i = pixel 2i+1, entry -1 = the left padding) and even pixels (entry i = pixel 2i, entry 128 = the right
//     padding).  Output pixel ow reads taps kw = 0..3 from odd[ow-1], even[ow], odd[ow], even[ow+1]: for the tap pairs
//     (0,1) and (2,3) that is start = odd[-1] / odd[0], row pitch 16 B, and the same plane distance + 16 B between the
//     two K chunks (lbo).  One K = 16 instruction per (kh, tap pair): 8 per output row.
//   CT = 4 (one source, 8 B per pixel): the row is staged shifted by one pixel, so the 16-byte entry ow holds pixels
//     (2ow-1, 2ow) and entry ow+1 holds (2ow+1, 2ow+2): start = entry 0, lbo = 16 B (overlapping core matrices).  One
//     K = 16 instruction per kh: 4 per output row.
// Input rows come in PAIRS (rows 2p-1, 2p; output row oh needs pairs oh and oh+1) through a ring of kTcSlots pair slots
// filled by cp.async (8-byte pieces, zero-filled outside the image), one stager warp per pair, four pairs in flight.
// Every CTA takes one contiguous range of output rows (two CTAs per SM).  Warp 0 issues the MMAs, warps 1-4 stage,
// warps 5-12 drain the accumulators (256 / cw TMEM stages): + bias, bf16, activation(s) into 128B-swizzled row tiles
// that leave through TMA stores (whole output rows, full lines).
// dynamic smem: out_s[2 rows][outputs][cw/64][128 px][128 B] | ws[16*CT/8][cw][16 B] | ring[kTcSlots][2 rows][kRowBytes] |
//               mbarriers | TMEM address
// ------------------------------------------------------------------------------------------------
constexpr int kTcSlots = 6;      // ring of row pairs (8320 B each for two sources)
constexpr int kTcPlane = 130 * 16;
constexpr int kTcStagers = 32;   // arrivals per staged pair: one stager warp (of four, warps 1-4) copies a whole pair
constexpr int kTcThreads = 416;  // warp 0 MMA | warps 1-4 staging | warps 5-12 epilogue (TMEM lane quarter = warp % 4;
                                 // two warps per quarter split each 64-column half: 4 warps were latency-bound)

template <int CT>
__global__ void __launch_bounds__(kTcThreads, 2) thin_conv_fwd_tc_kernel(const __grid_constant__ ThinFwdParams p) {
  constexpr int kRowBytes = (CT == 8 ? 2 : 1) * kTcPlane;
  constexpr int kSlotBytes = 2 * kRowBytes;
  constexpr int KC = 16 * CT / 8;            // 16-byte K chunks per weight row
  extern __shared__ uint8_t tc_raw[];
  const uint32_t base_a = (smem_u32(tc_raw) + 1023u) & ~1023u;
  uint8_t* base = tc_raw + (base_a - smem_u32(tc_raw));
  const int cw = p.cw;
  const int halves = cw >> 6;                // 64-channel output tiles per row
  const int outs_bytes = 2 * (p.out2 != nullptr ? 2 : 1) * halves * 16384;   // out_s[2 rows][outputs][halves][128 px][128 B], 128B-swizzled
  const int ws_bytes = KC * cw * 16;
  const uint32_t outs_a = base_a, ws_a = base_a + outs_bytes, ring_a = ws_a + ws_bytes;
  const uint32_t bar_a = ring_a + kTcSlots * kSlotBytes;
  uint8_t* ws = base + outs_bytes;
  volatile uint32_t* tmem_slot =
      reinterpret_cast<volatile uint32_t*>(ws + ws_bytes + kTcSlots * kSlotBytes + (2 * kTcSlots + 8) * 8);
  const int n_acc = 256 / cw;                // 4 (cw = 64) or 2 (cw = 128)
  auto pair_full = [&](int s) { return bar_a + s * 8; };
  auto pair_empty = [&](int s) { return bar_a + (kTcSlots + s) * 8; };
  auto acc_full = [&](int a) { return bar_a + (2 * kTcSlots + a) * 8; };
  auto acc_empty = [&](int a) { return bar_a + (2 * kTcSlots + 4 + a) * 8; };
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  // weights: ws[kc][n][8] <- w[n][kc*8 .. +8]   (core matrices of 8 output channels x 16 bytes)
  for (int idx = tid; idx < cw * KC; idx += kTcThreads) {
    const int n = idx / KC, kc = idx - n * KC;
    *reinterpret_cast<uint4*>(ws + (kc * cw + n) * 16) = ldg128(p.w + static_cast<long long>(n) * (16 * CT) + kc * 8);
  }
  for (int idx = tid; idx < kTcSlots * kSlotBytes / 16; idx += kTcThreads)      // padding entries stay zero for good
    *reinterpret_cast<uint4*>(ws + ws_bytes + idx * 16) = make_uint4(0, 0, 0, 0);
  if (tid == 0) {
    for (int s = 0; s < kTcSlots; ++s) {
      mbar_init(pair_full(s), kTcStagers);
      mbar_init(pair_empty(s), 1);
    }
    for (int a = 0; a < 4; ++a) {
      mbar_init(acc_full(a), 1);
      mbar_init(acc_empty(a), 8);
    }
    fence_mbar_init();
  }
  fence_proxy_async_smem();
  __syncthreads();
  if (warp == 0) {
    tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), 256);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // work split: every CTA takes one contiguous range of output rows (all images concatenated); a range is walked
  // in segments that stay inside one image (a segment of nrows output rows needs nrows + 1 row pairs)
  const int rows_total = p.n * p.oh;
  const int g_begin = static_cast<int>(static_cast<long long>(rows_total) * blockIdx.x / gridDim.x);
  const int g_end = static_cast<int>(static_cast<long long>(rows_total) * (blockIdx.x + 1) / gridDim.x);

  if (warp == 0) {
    // ------------------------------------------------------------------ MMA issue
    if (lane == 0) {
      const uint32_t idesc = make_idesc_bf16(128, cw, 0, 0);
      uint32_t c = 0, rs = 0;
      for (int g = g_begin; g < g_end;) {
        const int oh0 = g % p.oh;
        const int nrows = min(p.oh - oh0, g_end - g);
        g += nrows;
        for (int j = 0; j < nrows; ++j, ++rs) {
          const uint32_t a = rs % n_acc, aph = (rs / n_acc) & 1u;
          const uint32_t c0 = c + j;
          mbar_wait(acc_empty(a), aph ^ 1u);
          if (j == 0) mbar_wait(pair_full(c0 % kTcSlots), (c0 / kTcSlots) & 1u);   // (later rows saw it as c0 + 1)
          mbar_wait(pair_full((c0 + 1) % kTcSlots), ((c0 + 1) / kTcSlots) & 1u);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + a * cw;
#pragma unroll
          for (int kh = 0; kh < 4; ++kh) {
            const uint32_t cc = c0 + (kh >> 1);
            const uint32_t row_a = ring_a + (cc % kTcSlots) * kSlotBytes + (kh & 1) * kRowBytes;
            if (CT == 8) {
#pragma unroll
              for (int tp = 0; tp < 2; ++tp) {
                const uint64_t ad = make_nosw_desc(row_a + tp * 16, kTcPlane + 16, 128);
                const uint64_t bd = make_nosw_desc(ws_a + (kh * 4 + tp * 2) * cw * 16, cw * 16, 128);
                umma_bf16(d_tmem, ad, bd, idesc, (kh | tp) != 0);
              }
            } else {
              const uint64_t ad = make_nosw_desc(row_a, 16, 128);
              const uint64_t bd = make_nosw_desc(ws_a + (kh * 2) * cw * 16, cw * 16, 128);
              umma_bf16(d_tmem, ad, bd, idesc, kh != 0);
            }
          }
          umma_commit(acc_full(a));
          umma_commit(pair_empty(c0 % kTcSlots));                    // rows 2oh-1, 2oh are not needed again
          if (j == nrows - 1) umma_commit(pair_empty((c0 + 1) % kTcSlots));
        }
        c += nrows + 1;
      }
    }
  } else if (warp < 5) {
    // ------------------------------------------------------------------ staging
    // Stager warp sw copies the pairs whose running index is sw (mod 4), whole pairs on its own: cp.async, wait for ITS
    // copies, fence.proxy.async, 32 arrivals.  Four pairs are in flight per CTA without any thread having to fence
    // while younger copies are pending (a proxy fence waits for every outstanding cp.async of the thread, which
    // serialised a one-pair-per-iteration scheme at the memory latency).
    const int sw = warp - 1;
    const long long row_elems = static_cast<long long>(p.w_in) * 4;
    uint32_t c = 0;                            // running pair index
    for (int g = g_begin; g < g_end;) {
      const int img = g / p.oh;
      const int oh0 = g - img * p.oh;
      const int nrows = min(p.oh - oh0, g_end - g);
      g += nrows;
      const long long img_off = static_cast<long long>(img) * p.h * row_elems;
      for (int pj = 0; pj <= nrows; ++pj, ++c) {
        if ((c & 3u) != static_cast<uint32_t>(sw)) continue;
        const uint32_t slot = c % kTcSlots;
        mbar_wait(pair_empty(slot), ((c / kTcSlots) & 1u) ^ 1u);
        const int r0 = 2 * (oh0 + pj) - 1;
        const uint32_t dst0 = ring_a + slot * kSlotBytes;
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
          const int r = r0 + rr;
          const bool ok = static_cast<unsigned>(r) < static_cast<unsigned>(p.h) && !(p.skip & 4);
          const int nb = ok ? 8 : 0;
          const long long off_r = img_off + (ok ? r * row_elems : 0);
          const uint32_t d = dst0 + rr * kRowBytes;
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const int i = lane + 32 * t;       // pixels 2i (even) and 2i + 1 (odd)
            const long long off = off_r + i * 8;
            // CT = 8: even pixel -> even plane entry i, odd pixel -> odd plane entry i (entry -1 sits at byte 0)
            // CT = 4: pixel x at byte (x + 1) * 8
            const uint32_t d_even = CT == 8 ? kTcPlane + (i + 1) * 16 : (2 * i + 1) * 8;
            const uint32_t d_odd = CT == 8 ? (i + 1) * 16 : (2 * i + 2) * 8;
            cp_async8(d + d_even, p.s0 + off, nb);
            cp_async8(d + d_odd, p.s0 + off + 4, nb);
            if (CT == 8) {
              cp_async8(d + d_even + 8, p.s1 + off, nb);
              cp_async8(d + d_odd + 8, p.s1 + off + 4, nb);
            }
          }
        }
        cp_async_commit();
        cp_async_wait<0>();
        fence_proxy_async_smem();
        mbar_arrive(pair_full(slot));
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue
    // TMEM -> registers -> (+bias, bf16, activation(s)) -> 128B-swizzled smem row tiles -> TMA stores of whole output
    // rows (full lines; per-thread global stores of a pixel's 128 bytes made the store path the bottleneck).  One bulk
    // group per output row; the tiles are double-buffered by row parity.
    const int q = warp & 3;
    const int e_tid = tid - 160;               // 0 .. 255
    const int eh = (warp - 5) >> 2;            // which 32 columns of every 64-column half
    const int row = q * 32 + lane;             // pixel of the output row = TMEM lane
    const int n_pass = p.out2 != nullptr ? 2 : 1;
    const __nv_bfloat162 slope_a = __float2bfloat162_rn(p.slope1), slope_b = __float2bfloat162_rn(p.slope2);
    uint32_t rs = 0;
    for (int g = g_begin; g < g_end;) {
      const int img = g / p.oh;
      const int oh0 = g - img * p.oh;
      const int nrows = min(p.oh - oh0, g_end - g);
      g += nrows;
      for (int j = 0; j < nrows; ++j, ++rs) {
        const uint32_t a = rs % n_acc, aph = (rs / n_acc) & 1u;
        const uint32_t buf_a = outs_a + (rs & 1u) * n_pass * halves * 16384;     // [pass][half][128 px][128 B]
        mbar_wait(acc_full(a), aph);
        tc_fence_after();
        // the TMA stores that last read these tiles (two rows ago) have finished reading them
        if (e_tid == 0) tma_store_wait_read1();
        asm volatile("bar.sync 1, 256;" ::: "memory");
        const uint32_t t_row = tmem_base + a * cw + (static_cast<uint32_t>(q * 32) << 16);
        for (int hb = 0; hb < halves; ++hb) {
          uint32_t r[2][16];
#pragma unroll
          for (int i = 0; i < 2; ++i) tmem_ld16(t_row + hb * 64 + eh * 32 + i * 16, r[i]);
          tmem_ld_wait();
          if (hb == halves - 1) {                // accumulator drained: hand it back before the math
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(acc_empty(a));
          }
#pragma unroll
          for (int cl = 0; cl < 4; ++cl) {       // this warp's 16-byte chunks of the row's 128 bytes
            const int ch = eh * 4 + cl;
            float v[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) v[k] = __uint_as_float(r[cl >> 1][(cl & 1) * 8 + k]);
            if (p.bias != nullptr) {
              const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + hb * 64 + ch * 8));
              const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.bias + hb * 64 + ch * 8 + 4));
              v[0] += b0.x; v[1] += b0.y; v[2] += b0.z; v[3] += b0.w;
              v[4] += b1.x; v[5] += b1.y; v[6] += b1.z; v[7] += b1.w;
            }
            __nv_bfloat162 t[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) t[k] = __floats2bfloat162_rn(v[2 * k], v[2 * k + 1]);
            // act(v) = max(v, slope*v) for slope in [0, 1], on the packed bf16 pair (the tile kernel's arithmetic);
            // 16-byte chunk c of row r lives at chunk c ^ (r & 7) of the 128-byte row
            const uint32_t dst = buf_a + hb * 16384 + row * 128 + ((ch ^ (row & 7)) << 4);
#pragma unroll
            for (int pass = 0; pass < 2; ++pass) {
              if (pass == n_pass) break;
              const float slope = pass == 0 ? p.slope1 : p.slope2;
              const __nv_bfloat162 s2 = pass == 0 ? slope_a : slope_b;
              uint32_t pk[4];
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const __nv_bfloat162 u = slope != 1.f ? __hmax2(t[k], __hmul2(t[k], s2)) : t[k];
                pk[k] = *reinterpret_cast<const uint32_t*>(&u);
              }
              st_shared_v4(dst + pass * halves * 16384, pk[0], pk[1], pk[2], pk[3]);
            }
          }
        }
        fence_proxy_async_smem();
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (e_tid == 0 && !(p.skip & 2)) {
          for (int pass = 0; pass < n_pass; ++pass)
            for (int hb = 0; hb < halves; ++hb)
              tma_store_4d(&p.tm_row[pass], buf_a + (pass * halves + hb) * 16384, hb * 64, 0, oh0 + j, img);
          tma_store_commit();
        }
      }
    }
    if (e_tid == 0) tma_store_wait_all();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

// ------------------------------------------------------------------------------------------------
// Thin-input Conv2d(k4, s2, p1) weight gradient (and the last ConvTranspose2d's, with roles swapped):
//   dw[cw][tap][ch] += sum_pix wide[pix][cw] * thin[2*pix + tap - 1][ch];   dbias[cw] += sum_pix wide[pix][cw]
// wide = the 64/128-channel tensor at the coarse resolution (dY of the first convs, X of the last ConvT),
// thin = the 3-channel tensor(s) at twice the resolution (4 channel slots each).  K = pixels: per k-step one
// row of 16 coarse pixels; A fragments come from the wide tile with ldmatrix.trans, B fragments straight from
// the thin patch with ldmatrix.trans (a patch pixel is one 8/16-byte row of the im2col matrix that never
// exists).  CTA = persistent over 8 x 16 tiles with register accumulators, one atomic flush at the end.
// warp = (kernel row kh, 64-channel group).
// dynamic smem: patch[2][18][34][CT] | wide_s[2][128][cw + 8]   (bf16, cp.async double buffers)
// ------------------------------------------------------------------------------------------------
struct ThinWgradParams {
  CUtensorMap tm_wide;   // [n][oh][ow][cw] bf16: box 64 ch x 16 x 8 x 1, 128B swizzle, ragged tiles zero-filled
  CUtensorMap tm_row;    // the same tensor, box 64 ch x 128 x 1 x 1: one output row (tcgen05 row kernel)
  const bf16* wide;
  long long ld_w;
  const bf16* s0;
  long long ld0;
  const bf16* s1;
  long long ld1;
  int n, h, w_in, oh, ow, cw;
  float* dw;
  long long ld_m;
  int c_real;   // c0 + c1: channels per tap in the master layout
  int c0, c1;   // channels of source 0 / source 1 (slots 0..c0-1 and 4..4+c1-1 are real; the rest are dropped)
  float* dbias;
  int tiles_x, tiles_y;
  long long total_tiles;
};

template <int CT>
__global__ void __launch_bounds__(256) thin_conv_wgrad_kernel(const __grid_constant__ ThinWgradParams p) {
  constexpr int PW = CT / 2;
  constexpr int PATCH_WORDS = 18 * 34 * PW;
  constexpr int NT = CT / 2;             // n-tiles (8 columns) per kernel row: 4 taps * CT / 8
  // dynamic smem (1 KiB aligned): wide[2][cw/64][128 px][128 B] (TMA, 128B swizzle) | patch[2][18][34][CT] | 2 mbarriers
  extern __shared__ uint8_t dsm_raw[];
  const uint32_t wide_base = (smem_u32(dsm_raw) + 1023u) & ~1023u;
  uint8_t* dsm = dsm_raw + (wide_base - smem_u32(dsm_raw));
  const int wide_bytes = (p.cw >> 6) * 16384;          // one buffer
  uint32_t* patch_buf = reinterpret_cast<uint32_t*>(dsm + 2 * wide_bytes);
  const uint32_t bar0 = smem_u32(patch_buf + 2 * PATCH_WORDS);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int kh = warp & 3, mh = warp >> 2;
  const int nthr = blockDim.x;
  if (tid == 0) {
    tma_prefetch_desc(&p.tm_wide);
    mbar_init(bar0, 1);
    mbar_init(bar0 + 8, 1);
    fence_mbar_init();
  }
  __syncthreads();

  auto issue_tile = [&](long long tile, int buf) {
    const int t32 = static_cast<int>(tile), tpi = p.tiles_x * p.tiles_y;   // 32-bit: 64-bit division is ~10 % of the kernel
    const int img32 = t32 / tpi, rem32 = t32 - img32 * tpi;
    const int ty = rem32 / p.tiles_x, tx = rem32 - ty * p.tiles_x;
    const long long img = img32;
    const int oy0 = ty * 8, ox0 = tx * 16;
    const bf16* s0i = p.s0 + img * p.h * p.w_in * p.ld0;
    const bf16* s1i = CT == 8 ? p.s1 + img * p.h * p.w_in * p.ld1 : p.s0;
    const int ld0 = static_cast<int>(p.ld0), ld1 = static_cast<int>(p.ld1);
    const uint32_t dst0 = smem_u32(patch_buf + buf * PATCH_WORDS);
    for (int idx = tid; idx < 18 * 34; idx += nthr) {
      const int py = idx / 34, px = idx - py * 34;
      const int iy = 2 * oy0 - 1 + py, ix = 2 * ox0 - 1 + px;
      const bool ok = static_cast<unsigned>(iy) < static_cast<unsigned>(p.h) &&
                      static_cast<unsigned>(ix) < static_cast<unsigned>(p.w_in);
      const int pix = ok ? iy * p.w_in + ix : 0;
      cp_async8(dst0 + idx * PW * 4, s0i + pix * ld0, ok ? 8 : 0);
      if (CT == 8) cp_async8(dst0 + idx * PW * 4 + 8, s1i + pix * ld1, ok ? 8 : 0);
    }
    // the wide tile (dY / X at the coarse resolution) comes by TMA: the per-thread cp.async loop was 16 % of the
    // kernel's instructions; pixels outside the image are zero-filled by the unit
    if (tid == 0) {
      const uint32_t bar = bar0 + 8 * buf;
      mbar_expect_tx(bar, static_cast<uint32_t>(wide_bytes));
      for (int b = 0; b < (p.cw >> 6); ++b)
        tma_load_4d(wide_base + buf * wide_bytes + b * 16384, &p.tm_wide, bar, b * 64, ox0, oy0, img32);
    }
    cp_async_commit();
  };

  float acc[4][NT][4];
  float accb[4][4];
#pragma unroll
  for (int mi = 0; mi < 4; ++mi) {
#pragma unroll
    for (int ni = 0; ni < NT; ++ni)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[mi][ni][j] = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) accb[mi][j] = 0.f;
  }
  const bool do_bias = p.dbias != nullptr && kh == 0;

  if (static_cast<long long>(blockIdx.x) < p.total_tiles) issue_tile(blockIdx.x, 0);
  int buf = 0;
  uint32_t wphase[2] = {0u, 0u};
  for (long long tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, buf ^= 1) {
    const long long next = tile + gridDim.x;
    __syncthreads();  // everyone finished reading buffer buf^1 (previous tile)
    if (next < p.total_tiles) {
      issue_tile(next, buf ^ 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    mbar_wait(bar0 + 8 * buf, wphase[buf]);
    wphase[buf] ^= 1u;
    __syncthreads();
    const uint32_t patch_a = smem_u32(patch_buf + buf * PATCH_WORDS);
    const uint32_t wide_a = wide_base + buf * wide_bytes + mh * 16384;
#pragma unroll 2
    for (int r = 0; r < 8; ++r) {     // k-step: output row r of the tile, 16 pixels
      // A (m = channels, k = pixels): wide_s[px][cw] read transposed
      uint32_t a[4][4];
#pragma unroll
      for (int mi = 0; mi < 4; ++mi) {
        const int px = r * 16 + (lane & 7) + ((lane >> 4) << 3);
        const int chunk = mi * 2 + ((lane >> 3) & 1);          // 16-byte chunk of the 64-channel row (128B swizzle)
        ldmatrix_x4_trans(a[mi], wide_a + px * 128 + ((chunk ^ (px & 7)) << 4));
      }
      // B (k = pixels, n = (tap, slot)): patch pixels (2r + kh, 2*ox + kw) are the rows
#pragma unroll
      for (int ni = 0; ni < NT; ++ni) {
        // CT = 8: n-tile = tap kw = ni (16 B per pixel);  CT = 4: n-tile = taps kw = 2ni, 2ni+1 (two 8 B pixels)
        const int kw = CT == 8 ? ni : 2 * ni;
        const int ox = lane & 15;
        uint32_t b0, b1;
        ldmatrix_x2_trans(b0, b1, patch_a + (((2 * r + kh) * 34 + 2 * ox + kw) * PW) * 4);
#pragma unroll
        for (int mi = 0; mi < 4; ++mi) mma_bf16_16816(acc[mi][ni], a[mi], b0, b1);
      }
      if (do_bias) {
#pragma unroll
        for (int mi = 0; mi < 4; ++mi) mma_bf16_16816(accb[mi], a[mi], 0x3F803F80u, 0x3F803F80u);
      }
    }
  }

  // flush: rows = channels mh*64 + mi*16 + g (+8); columns n = ni*8 + 2t (+1) -> (tap, slot)
#pragma unroll
  for (int mi = 0; mi < 4; ++mi) {
    const int c0 = mh * 64 + mi * 16 + g;
#pragma unroll
    for (int ni = 0; ni < NT; ++ni) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int ncol = 2 * t + e;
        int tap, slot;
        if (CT == 8) {
          tap = kh * 4 + ni;
          slot = ncol;
        } else {
          tap = kh * 4 + 2 * ni + (ncol >> 2);
          slot = ncol & 3;
        }
        if ((slot & 3) >= (slot < 4 ? p.c0 : p.c1)) continue;
        const int ch = slot < 4 ? slot : p.c0 + slot - 4;
        atomicAdd(p.dw + static_cast<long long>(c0) * p.ld_m + tap * p.c_real + ch, acc[mi][ni][e]);
        atomicAdd(p.dw + static_cast<long long>(c0 + 8) * p.ld_m + tap * p.c_real + ch, acc[mi][ni][2 + e]);
      }
    }
    if (do_bias && t == 0) {
      atomicAdd(p.dbias + c0, accb[mi][0]);
      atomicAdd(p.dbias + c0 + 8, accb[mi][2]);
    }
  }
}


// ------------------------------------------------------------------------------------------------
// The same weight gradient on tcgen05 for 256-pixel rows (dense 4-slot sources):
//   D[m][co] += sum_ow  A[m][ow] * dy[ow][co],   m = (kh*4 + kw)*CT + slot   (A = the im2col matrix, transposed)
// accumulated in ONE TMEM tile over all the output rows a CTA owns (K = pixels) and flushed with atomics at the end.
// Both operands are MN-major: dy rows arrive by TMA as 128B-swizzled [128 px][64 co] tiles, and A is read straight
// out of staged copies of the image rows through an un-swizzled MN-major descriptor -- 16-byte M chunks `sbo` apart,
// eight consecutive ow 16 bytes apart.  A chunk is one (kh, kw) tap of the concatenated 8-slot pixel (CT = 8) or one
// (kh, pixel pair) of the single source (CT = 4); a uniform chunk pitch needs every x row staged as four (two) shifted
// planes of 128 entries: plane kw, entry ow = pixel 2ow - 1 + kw (CT = 8); plane ps, entry ow = pixels 2ow - 1 + 2ps,
// 2ow + 2ps (CT = 4).  Rows are staged in PAIRS (rows 2p-1, 2p = kh 0,1 of output row p and kh 2,3 of row p-1) into a
// ring of four 8-plane slots; an output row reads two consecutive slots with one descriptor, so the pair that lands
// in slot 0 is also written to a mirror slot behind slot 3.  CT = 4 has only 64 valid M rows: the upper 64 TMEM lanes
// accumulate whatever follows in shared memory and are never read.
// Warp 0 issues the MMAs (8 per output row), warps 1-4 stage x (cp.async, one warp per pair), warp 5 issues the dy
// TMA loads, warps 6-9 sum the dy tiles for the bias gradient and flush the accumulator at the end.
// dynamic smem (1 KiB aligned): dy_s[4][cw/64][128 px][128 B] | ring[(5 + 3) slots][8 planes][2 KiB (CT/8)] | mbarriers |
//                               bias partial sums [2][16][64] fp32
// ------------------------------------------------------------------------------------------------
constexpr int kWtThreads = 320;
constexpr int kWtSlots = 4;

template <int CT>
__global__ void __launch_bounds__(kWtThreads, 1) thin_conv_wgrad_tc_kernel(const __grid_constant__ ThinWgradParams p) {
  constexpr int kPlane = 2048;                           // 128 entries x 16 B
  constexpr int kPlanesPerRow = CT == 8 ? 4 : 2;
  constexpr int kSlotBytes = 2 * kPlanesPerRow * kPlane;   // one pair of x rows
  constexpr int kRingSlots = kWtSlots + 1 + 3;           // + mirror of slot 0 + slack the CT = 4 descriptor runs into
  extern __shared__ uint8_t wt_raw[];
  const uint32_t base_a = (smem_u32(wt_raw) + 1023u) & ~1023u;
  uint8_t* base = wt_raw + (base_a - smem_u32(wt_raw));
  const int cw = p.cw, halves = cw >> 6;
  const int dy_bytes = halves * 16384;
  const uint32_t dy_a = base_a, ring_a = base_a + 4 * dy_bytes;
  const uint32_t bar_a = ring_a + kRingSlots * kSlotBytes;
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(base + 4 * dy_bytes + kRingSlots * kSlotBytes + 20 * 8);
  auto xfull = [&](int s) { return bar_a + s * 8; };
  auto xempty = [&](int s) { return bar_a + (4 + s) * 8; };
  auto dfull = [&](int s) { return bar_a + (8 + s) * 8; };
  auto dempty = [&](int s) { return bar_a + (12 + s) * 8; };
  const uint32_t acc_done = bar_a + 16 * 8;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool do_bias = p.dbias != nullptr;

  for (int idx = tid; idx < kRingSlots * kSlotBytes / 16; idx += kWtThreads)      // edge entries stay zero for good
    *reinterpret_cast<uint4*>(base + 4 * dy_bytes + idx * 16) = make_uint4(0, 0, 0, 0);
  if (tid == 0) {
    for (int s2 = 0; s2 < 4; ++s2) {
      mbar_init(xfull(s2), 32);
      mbar_init(xempty(s2), 1);
      mbar_init(dfull(s2), 1);
      mbar_init(dempty(s2), do_bias ? 5 : 1);
    }
    mbar_init(acc_done, 1);
    fence_mbar_init();
  }
  fence_proxy_async_smem();
  __syncthreads();
  if (warp == 0) {
    tmem_alloc(smem_u32(const_cast<uint32_t*>(tmem_slot)), 128);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int rows_total = p.n * p.oh;
  const int g_begin = static_cast<int>(static_cast<long long>(rows_total) * blockIdx.x / gridDim.x);
  const int g_end = static_cast<int>(static_cast<long long>(rows_total) * (blockIdx.x + 1) / gridDim.x);

  if (warp == 0) {
    // ------------------------------------------------------------------ MMA issue
    if (lane == 0) {
      const uint32_t idesc = make_idesc_bf16(128, cw, 1, 1);
      uint32_t c = 0, rs = 0;
      for (int g = g_begin; g < g_end;) {
        const int oh0 = g % p.oh;
        const int nrows = min(p.oh - oh0, g_end - g);
        g += nrows;
        for (int j = 0; j < nrows; ++j, ++rs) {
          const uint32_t c0 = c + j, s0 = c0 & 3u;      // pairs c0, c0 + 1 sit in slots s0, s0 + 1 (mirror when s0 = 3)
          if (j == 0) mbar_wait(xfull(s0), (c0 >> 2) & 1u);
          mbar_wait(xfull((c0 + 1) & 3u), ((c0 + 1) >> 2) & 1u);
          mbar_wait(dfull(rs & 3u), (rs >> 2) & 1u);
          tc_fence_after();
          const uint32_t a_row = ring_a + s0 * kSlotBytes, b_row = dy_a + (rs & 3u) * dy_bytes;
#pragma unroll
          for (int k = 0; k < 8; ++k) {                  // 16 output pixels per instruction
            const uint64_t ad = make_nosw_desc(a_row + k * 256, 128, kPlane);
            const uint64_t bd = make_sw128_desc(b_row + k * 2048, 16384, 1024);
            umma_bf16(tmem_base, ad, bd, idesc, (rs | k) != 0);
          }
          umma_commit(xempty(s0));                       // rows 2oh-1, 2oh are not needed again
          if (j == nrows - 1) umma_commit(xempty((c0 + 1) & 3u));
          umma_commit(dempty(rs & 3u));
        }
        c += nrows + 1;
      }
      umma_commit(acc_done);
    }
  } else if (warp < 5) {
    // ------------------------------------------------------------------ x staging: one warp per pair
    const int sw = warp - 1;
    const long long row_elems = static_cast<long long>(p.w_in) * 4;
    uint32_t c = 0;
    for (int g = g_begin; g < g_end;) {
      const int img = g / p.oh;
      const int oh0 = g - img * p.oh;
      const int nrows = min(p.oh - oh0, g_end - g);
      g += nrows;
      const long long img_off = static_cast<long long>(img) * p.h * row_elems;
      for (int pj = 0; pj <= nrows; ++pj, ++c) {
        if ((c & 3u) != static_cast<uint32_t>(sw)) continue;
        const uint32_t slot = c & 3u;
        mbar_wait(xempty(slot), ((c >> 2) & 1u) ^ 1u);
        const int r0 = 2 * (oh0 + pj) - 1;
        for (int copy = 0; copy < ((slot == 0 && c > 0) ? 2 : 1); ++copy) {
          const uint32_t dst0 = ring_a + (copy ? kWtSlots : slot) * kSlotBytes;
#pragma unroll
          for (int rr = 0; rr < 2; ++rr) {
            const int r = r0 + rr;
            const bool ok = static_cast<unsigned>(r) < static_cast<unsigned>(p.h);
            const int nb = ok ? 8 : 0;
            const long long off_r = img_off + (ok ? r * row_elems : 0);
            const uint32_t d = dst0 + rr * kPlanesPerRow * kPlane;
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              const int i = lane + 32 * t;               // pixels 2i (even) and 2i + 1 (odd)
              const long long off = off_r + i * 8;
              if (CT == 8) {
                // even pixel 2i: plane 1 entry i, plane 3 entry i-1; odd pixel 2i+1: plane 0 entry i+1, plane 2 entry i
                cp_async8(d + 1 * kPlane + i * 16, p.s0 + off, nb);
                cp_async8(d + 1 * kPlane + i * 16 + 8, p.s1 + off, nb);
                if (i > 0) {
                  cp_async8(d + 3 * kPlane + (i - 1) * 16, p.s0 + off, nb);
                  cp_async8(d + 3 * kPlane + (i - 1) * 16 + 8, p.s1 + off, nb);
                }
                if (i < 127) {
                  cp_async8(d + 0 * kPlane + (i + 1) * 16, p.s0 + off + 4, nb);
                  cp_async8(d + 0 * kPlane + (i + 1) * 16 + 8, p.s1 + off + 4, nb);
                }
                cp_async8(d + 2 * kPlane + i * 16, p.s0 + off + 4, nb);
                cp_async8(d + 2 * kPlane + i * 16 + 8, p.s1 + off + 4, nb);
              } else {
                // plane ps, entry e = pixels (2e-1+2ps, 2e+2ps): even pixel 2i -> second half of (0, i) and (1, i-1);
                // odd pixel 2i+1 -> first half of (0, i+1) and (1, i)
                cp_async8(d + 0 * kPlane + i * 16 + 8, p.s0 + off, nb);
                if (i > 0) cp_async8(d + 1 * kPlane + (i - 1) * 16 + 8, p.s0 + off, nb);
                if (i < 127) cp_async8(d + 0 * kPlane + (i + 1) * 16, p.s0 + off + 4, nb);
                cp_async8(d + 1 * kPlane + i * 16, p.s0 + off + 4, nb);
              }
            }
          }
        }
        cp_async_commit();
        cp_async_wait<0>();
        fence_proxy_async_smem();
        mbar_arrive(xfull(slot));
      }
    }
  } else if (warp == 5) {
    // ------------------------------------------------------------------ dy rows by TMA
    if (lane == 0) {
      uint32_t rs = 0;
      for (int g = g_begin; g < g_end; ++g, ++rs) {
        const int img = g / p.oh, oh = g - img * p.oh;
        const uint32_t slot = rs & 3u;
        mbar_wait(dempty(slot), ((rs >> 2) & 1u) ^ 1u);
        mbar_expect_tx(dfull(slot), dy_bytes);
        for (int hb = 0; hb < halves; ++hb)
          tma_load_4d(dy_a + slot * dy_bytes + hb * 16384, &p.tm_row, dfull(slot), hb * 64, 0, oh, img);
      }
    }
  } else {
    // ------------------------------------------------------------------ bias sums per row, accumulator flush at the end
    const int q = warp & 3;
    const int e_tid = tid - 192;               // 0 .. 127
    // thread -> 16-byte column chunk it always reads (the swizzle XOR is constant along its pixels r0 + 16 i)
    const int r0 = e_tid >> 3, chunk = (e_tid & 7) ^ (r0 & 7);
    float bs[2][8];
#pragma unroll
    for (int hb = 0; hb < 2; ++hb)
#pragma unroll
      for (int k = 0; k < 8; ++k) bs[hb][k] = 0.f;
    if (do_bias) {
      uint32_t rs = 0;
      for (int g = g_begin; g < g_end; ++g, ++rs) {
        const uint32_t slot = rs & 3u;
        mbar_wait(dfull(slot), (rs >> 2) & 1u);
        const uint8_t* tile = base + slot * dy_bytes;
#pragma unroll
        for (int hb = 0; hb < 2; ++hb) {       // (static bounds: bs[][] must stay in registers)
          if (hb >= halves) break;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const uint4 raw = *reinterpret_cast<const uint4*>(tile + hb * 16384 + (r0 + 16 * i) * 128 + (e_tid & 7) * 16);
            const uint32_t w4[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              bs[hb][2 * k] += bf16_lo(w4[k]);
              bs[hb][2 * k + 1] += bf16_hi(w4[k]);
            }
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(dempty(slot));
      }
      // 16 threads (r0 = 0 .. 15) hold partial sums of the same 8 channels: combine them in shared memory so that every
      // CTA adds ONE value per channel (16 x 148 same-address atomics per channel cost more than the whole kernel)
      float* red = reinterpret_cast<float*>(base + 4 * dy_bytes + kRingSlots * kSlotBytes + 32 * 8);   // [2][16][64]
#pragma unroll
      for (int hb = 0; hb < 2; ++hb) {
        if (hb >= halves) break;
#pragma unroll
        for (int k = 0; k < 8; ++k) red[(hb * 16 + r0) * 64 + chunk * 8 + k] = bs[hb][k];
      }
      asm volatile("bar.sync 2, 128;" ::: "memory");
      for (int col = e_tid; col < cw; col += 128) {
        const int hb = col >> 6, cc = col & 63;
        float tot = 0.f;
#pragma unroll
        for (int r = 0; r < 16; ++r) tot += red[(hb * 16 + r) * 64 + cc];
        atomicAdd(p.dbias + col, tot);
      }
    }
    if (g_end > g_begin) {
      mbar_wait(acc_done, 0u);
      tc_fence_after();
      const int m = q * 32 + lane;             // TMEM lane = im2col row
      int tap, ch;
      bool valid;
      if (CT == 8) {
        const int s8 = m & 7;
        tap = m >> 3;
        valid = (s8 & 3) < (s8 < 4 ? p.c0 : p.c1);
        ch = s8 < 4 ? s8 : p.c0 + s8 - 4;
      } else {
        const int s4 = m & 3;
        tap = m >> 2;
        valid = m < 64 && s4 < p.c0;
        ch = s4;
      }
      float* dst = p.dw + tap * p.c_real + ch;
      for (int c0 = 0; c0 < cw; c0 += 16) {
        uint32_t r[16];
        tmem_ld16(tmem_base + c0 + (static_cast<uint32_t>(q * 32) << 16), r);
        tmem_ld_wait();
        if (valid) {
#pragma unroll
          for (int k = 0; k < 16; ++k) atomicAdd(dst + static_cast<long long>(c0 + k) * p.ld_m, __uint_as_float(r[k]));
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 128);
  }
}

// ------------------------------------------------------------------------------------------------
// Thin-output ConvTranspose2d(cw -> CO, k4, s2, p1), CO = 1..4: the generator's last layer (+bias, Tanh;
// models.py:184,186) and the input gradient of the discriminator's first conv (once per source).  Per CTA: a 10 x 18
// halo tile of `wide` (8 x 16 source pixels + 1 ring) is multiplied by wcol[16*CO = tap*CO + co][cw] into
// col[halo pixel][16*CO] (fp32, shared memory) with warp MMAs, then every output pixel of the 16 x 32 output tile
// sums its 4 taps (col2im inside the CTA; the ring makes the tile self-contained), adds the bias, applies Tanh and is
// written once; output slots >= CO are written as zero.
// The halo tile arrives by TMA (one 4-D box per 64 channels, out-of-range pixels zero-filled): the per-thread
// cp.async loop it replaces was 40 % of the kernel's instructions (ncu source page), on an issue-bound kernel.
// dynamic smem (1 KiB aligned): wide_s[cw/64][192 rows][128 B] (bf16, 128B-swizzled TMA tiles) | w_s[16*CO][cw+8] (bf16) |
//                               col_s[192][thin_convT_col_stride(CO)] (fp32) | mbarrier
// ------------------------------------------------------------------------------------------------
struct ThinConvTParams {
  CUtensorMap tm_wide;   // [n][ih][iw][cw] bf16, box 64 ch x 18 x 10 x 1, 128B swizzle, OOB = zero (the halo ring)
  const bf16* wide;
  long long ld_w;
  const bf16* wcol;
  const float* bias;
  int n, ih, iw, cw, act;
  bf16* out_bf;
  long long ld_bf;
  float* out_f32;
  long long ld_f;
  uint8_t* out_u8;   // [n][2ih][2iw][CO]: uint8((v*0.5 + 0.5) * 255), the image generate_synthetic_data.py:69-88 saves
  int tiles_x, tiles_y;
  long long total_tiles;
};

// fp32 per col_s row (16*CO used).  In a warp the col2im reads 16 neighbouring halo pixels at one tap column (even
// lanes) and the next 16 at the column CO lower (odd lanes).  CO = 3: 50 = 18 mod 32 puts the even lanes on the 16 even
// banks and the odd lanes on the odd ones; CO = 1 likewise with 18.  CO = 2 / 4 read each tap as one float2 / float4:
// a stride of 18 vectors keeps the 16 (8) lanes of one shared-memory wavefront on distinct 8 (16) byte slots.
__host__ __device__ constexpr int thin_convT_col_stride(int co) { return co == 3 ? 50 : 18 * co; }

constexpr int kWideBoxRows = 180;               // 10 x 18 halo pixels per box
constexpr int kWideTileBytes = 192 * 128;       // one 64-channel tile: 192 MMA rows (180 loaded, 12 kept zero)

// tanh through one exp and one fast division: absolute error ~1e-7 (the output is an image in [-1, 1]; the libdevice
// tanhf it replaces cost 12 % of the kernel's instructions).
__device__ __forceinline__ float tanh_fast(float x) {
  const float e = __expf(2.f * x);              // inf for large x -> 1, 0 for very negative x -> -1
  return 1.f - __fdividef(2.f, e + 1.f);
}

template <int CO>
__global__ void __launch_bounds__(256) thin_convT_fwd_kernel(const __grid_constant__ ThinConvTParams p) {
  constexpr int NCOL = 16 * CO;                  // (tap, co) columns
  constexpr int NT = CO;                         // 8-column n-tiles per warp (a warp owns half of the columns)
  constexpr int kColStride = thin_convT_col_stride(CO);
  extern __shared__ uint8_t dsm_raw[];
  const uint32_t wide_a = (smem_u32(dsm_raw) + 1023u) & ~1023u;
  uint8_t* dsm = dsm_raw + (wide_a - smem_u32(dsm_raw));
  const int wstride = p.cw + 8;
  const int nbox = p.cw >> 6;
  bf16* w_s = reinterpret_cast<bf16*>(dsm + nbox * kWideTileBytes);
  float* col_s = reinterpret_cast<float*>(w_s + NCOL * wstride);
  const uint32_t bar = smem_u32(col_s + 192 * kColStride);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int vshift = p.cw == 64 ? 3 : 4;
  const int oh = 2 * p.ih, ow = 2 * p.iw;
  const int mg = warp >> 1, nh = warp & 1;   // warp = 3 m-tiles (48 halo pixels) x NT n-tiles (8*NT columns)

  if (tid == 0) {
    tma_prefetch_desc(&p.tm_wide);
    mbar_init(bar, 1);
    fence_mbar_init();
  }
  // MMA rows 180..191 of every tile are never written by the TMA box: keep them zero
  for (int idx = tid; idx < nbox * 12 * 8; idx += 256) {
    const int b = idx / 96, r = (idx % 96) >> 3, seg = idx & 7;
    *reinterpret_cast<uint4*>(dsm + b * kWideTileBytes + (kWideBoxRows + r) * 128 + seg * 16) = make_uint4(0, 0, 0, 0);
  }
  for (int idx = tid; idx < (NCOL << vshift); idx += 256) {
    const int r = idx >> vshift, seg = idx & ((1 << vshift) - 1);
    *reinterpret_cast<uint4*>(w_s + r * wstride + seg * 8) = ldg128(p.wcol + static_cast<long long>(r) * p.cw + seg * 8);
  }
  float biasv[CO];
#pragma unroll
  for (int j = 0; j < CO; ++j) biasv[j] = p.bias != nullptr ? __ldg(p.bias + j) : 0.f;
  const uint32_t w_a = smem_u32(w_s);
  const int kchunks = p.cw >> 4;
  const int tiles_per_img = p.tiles_x * p.tiles_y;
  uint32_t phase = 0;

  // tid 0 issues the halo-tile load of `tile`; it runs one tile ahead: the next load is issued as soon as the MMA
  // phase has finished reading wide_s and overlaps the col2im phase (which only reads col_s)
  auto issue_load = [&](int tile) {
    const int img = tile / tiles_per_img, rem = tile - img * tiles_per_img;
    const int ty = rem / p.tiles_x, tx = rem - ty * p.tiles_x;
    mbar_expect_tx(bar, static_cast<uint32_t>(nbox * kWideBoxRows * 128));
    for (int b = 0; b < nbox; ++b)
      tma_load_4d(wide_a + b * kWideTileBytes, &p.tm_wide, bar, b * 64, tx * 16 - 1, ty * 8 - 1, img);
  };
  const int total = static_cast<int>(p.total_tiles);
  __syncthreads();  // w_s, the zero rows and the barrier are set up
  if (tid == 0 && static_cast<int>(blockIdx.x) < total) issue_load(blockIdx.x);

  for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
    const int img = tile / tiles_per_img, rem = tile - img * tiles_per_img;
    const int ty = rem / p.tiles_x, tx = rem - ty * p.tiles_x;
    const int i0 = ty * 8, j0 = tx * 16;
    mbar_wait(bar, phase);
    phase ^= 1u;
    // ---- col = wide_s (192 x cw) * wcol^T (cw x 16*CO)
    float acc[3][NT][4];
#pragma unroll
    for (int mi = 0; mi < 3; ++mi)
#pragma unroll
      for (int ni = 0; ni < NT; ++ni)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[mi][ni][j] = 0.f;
    for (int kc = 0; kc < kchunks; ++kc) {
      uint32_t a[3][4], b[NT][2];
#pragma unroll
      for (int mi = 0; mi < 3; ++mi) {
        // 128B-swizzled tile: 16-byte chunk c of row r lives at chunk (c ^ (r & 7))
        const int row = (mg * 3 + mi) * 16 + (lane & 15);
        const int chunk = ((kc & 3) << 1) + (lane >> 4);
        ldmatrix_x4(a[mi], wide_a + (kc >> 2) * kWideTileBytes + row * 128 + ((chunk ^ (row & 7)) << 4));
      }
      // B fragments: pairs of n-tiles with one x4 load, an odd last n-tile with an x2 load
#pragma unroll
      for (int ni = 0; ni + 1 < NT; ni += 2) {
        uint32_t r4[4];
        ldb_16x16(r4, w_a + ((nh * NT + ni) * 8 * wstride + kc * 16) * 2, wstride * 2, lane);
        b[ni][0] = r4[0];
        b[ni][1] = r4[1];
        b[ni + 1][0] = r4[2];
        b[ni + 1][1] = r4[3];
      }
      if (NT & 1)
        ldmatrix_x2(b[NT - 1][0], b[NT - 1][1],
                    w_a + (((nh * NT + NT - 1) * 8 + (lane & 7)) * wstride + kc * 16 + ((lane >> 3) & 1) * 8) * 2);
#pragma unroll
      for (int mi = 0; mi < 3; ++mi)
#pragma unroll
        for (int ni = 0; ni < NT; ++ni) mma_bf16_16816(acc[mi][ni], a[mi], b[ni][0], b[ni][1]);
    }
#pragma unroll
    for (int mi = 0; mi < 3; ++mi) {
      const int px0 = (mg * 3 + mi) * 16 + g;
#pragma unroll
      for (int ni = 0; ni < NT; ++ni) {
        const int col = (nh * NT + ni) * 8 + 2 * t;
        *reinterpret_cast<float2*>(col_s + px0 * kColStride + col) = make_float2(acc[mi][ni][0], acc[mi][ni][1]);
        *reinterpret_cast<float2*>(col_s + (px0 + 8) * kColStride + col) = make_float2(acc[mi][ni][2], acc[mi][ni][3]);
      }
    }
    __syncthreads();   // col_s complete; nobody reads wide_s any more
    if (tid == 0 && tile + static_cast<int>(gridDim.x) < total) issue_load(tile + gridDim.x);
    // ---- col2im inside the tile: output (yl, xl) sums its 2 x 2 taps
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int pix = tid + k * 256, yl = pix >> 5, xl = pix & 31;
      const int y = 2 * i0 + yl, x = 2 * j0 + xl;
      if (y >= oh || x >= ow) continue;
      float v[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int j = 0; j < CO; ++j) v[j] = biasv[j];
#pragma unroll
      for (int a2 = 0; a2 < 2; ++a2) {
        const int kh = ((yl + 1) & 1) + 2 * a2;          // taps with (yl + 1 - kh) even
        const int r = ((yl + 1 - kh) >> 1) + 1;          // halo row of the source pixel
#pragma unroll
        for (int b2 = 0; b2 < 2; ++b2) {
          const int kw = ((xl + 1) & 1) + 2 * b2;
          const int c = ((xl + 1 - kw) >> 1) + 1;
          const float* src = col_s + (r * 18 + c) * kColStride + (kh * 4 + kw) * CO;
          if constexpr (CO == 4) {
            const float4 q = *reinterpret_cast<const float4*>(src);
            v[0] += q.x;
            v[1] += q.y;
            v[2] += q.z;
            v[3] += q.w;
          } else if constexpr (CO == 2) {
            const float2 q = *reinterpret_cast<const float2*>(src);
            v[0] += q.x;
            v[1] += q.y;
          } else {
#pragma unroll
            for (int j = 0; j < CO; ++j) v[j] += src[j];
          }
        }
      }
      if (p.act == GAP_ACT_TANH) {
#pragma unroll
        for (int j = 0; j < CO; ++j) v[j] = tanh_fast(v[j]);
      }
      const long long o = (static_cast<long long>(img) * oh + y) * ow + x;
      if (p.out_f32) *reinterpret_cast<float4*>(p.out_f32 + o * p.ld_f) = make_float4(v[0], v[1], v[2], v[3]);
      if (p.out_bf) *reinterpret_cast<uint2*>(p.out_bf + o * p.ld_bf) = make_uint2(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]));
      if (p.out_u8) {
#pragma unroll
        for (int j = 0; j < CO; ++j) {
          const float u = fminf(fmaxf((v[j] * 0.5f + 0.5f) * 255.f, 0.f), 255.f);
          p.out_u8[o * CO + j] = static_cast<uint8_t>(u);   // truncation, like torchvision's to_pil_image (mul(255).byte())
        }
      }
    }
    __syncthreads();   // col_s is free for the next tile
  }
}

// BCE-with-logits against a constant target with an fp32 gradient and the bias gradient of the
// producing Cout = 1 conv:  dlogits = grad_scale*(sigmoid(x) - t);  dbias += sum dlogits
__global__ void bce_logits_const_f32_kernel(const float* __restrict__ x, long long count, float t, float grad_scale,
                                            float* __restrict__ dx, double* __restrict__ loss_acc,
                                            float* __restrict__ dbias) {
  float part = 0.f, gsum = 0.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < count;
       i += (long long)gridDim.x * blockDim.x) {
    const float v = x[i];
    part += fmaxf(v, 0.f) - v * t + log1pf(__expf(-fabsf(v)));
    const float d = grad_scale * (1.f / (1.f + __expf(-v)) - t);
    if (dx) dx[i] = d;
    gsum += d;
  }
  part = warp_sum(part);
  gsum = warp_sum(gsum);
  __shared__ float red[2][32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) {
    red[0][wid] = part;
    red[1][wid] = gsum;
  }
  __syncthreads();
  if (wid == 0) {
    float v = lane < (blockDim.x >> 5) ? red[0][lane] : 0.f;
    float gg = lane < (blockDim.x >> 5) ? red[1][lane] : 0.f;
    v = warp_sum(v);
    gg = warp_sum(gg);
    if (lane == 0) {
      atomicAdd(loss_acc, static_cast<double>(v));
      if (dbias) atomicAdd(dbias, gg);
    }
  }
}

// uint8 HWC image [pixel][C] -> normalised NHWC bf16 with 4 channel slots: (x/255 - 0.5)/0.5 (dataset.py:155-159 on the
// device); slots >= C are written as zero
template <int C>
__global__ void u8_hwc_to_nhwc_bf16_kernel(const uint8_t* __restrict__ x, bf16* __restrict__ out, long long ld,
                                           long long pixels) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < pixels; i += (long long)gridDim.x * blockDim.x) {
    float v[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int j = 0; j < C; ++j) v[j] = x[i * C + j] * (2.f / 255.f) - 1.f;
    *reinterpret_cast<uint2*>(out + i * ld) = make_uint2(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]));
  }
}

// ------------------------------------------------------------------------------------------------
// dataset.py's JointResize + JointNormalize on the device (dataset.py:136-159): uint8 HWC image -> bilinear resize of
// the [0, 1] tensor -> x*2 - 1 -> NHWC bf16 with 4 channel slots.  The reference resizes TENSORS with
// torchvision.transforms.functional.resize(BILINEAR), i.e. F.interpolate(mode="bilinear", align_corners=False,
// antialias=True): a separable triangle filter whose support grows with the down-scaling factor (ATen
// upsample_bilinear2d_aa; identical to plain bilinear when up-scaling).  Per output index i along an axis:
//   scale = in / out; support = max(scale, 1); center = scale * (i + 0.5)
//   taps j in [max(0, int(center - support + 0.5)), min(in, int(center + support + 0.5)));
//   w_j = max(0, 1 - |(j - center + 0.5) / max(scale, 1)|), normalised to sum 1.
// One thread per output pixel, all C channels (1..4; slots >= C of the bf16 output are written as zero); the 2-D weights
// are the product of the two 1-D ones.
// ------------------------------------------------------------------------------------------------
struct AaAxis {
  int lo, n;
  float center, inv, total;
};
__device__ __forceinline__ AaAxis aa_axis(int i, int in, float scale) {
  AaAxis a;
  const float support = fmaxf(scale, 1.f);
  a.center = scale * (i + 0.5f);
  a.inv = 1.f / support;
  a.lo = max(0, static_cast<int>(a.center - support + 0.5f));
  a.n = min(in, static_cast<int>(a.center + support + 0.5f)) - a.lo;
  a.total = 0.f;
  for (int j = 0; j < a.n; ++j) a.total += fmaxf(0.f, 1.f - fabsf((j + a.lo - a.center + 0.5f) * a.inv));
  return a;
}
template <int C>
__global__ void resize_u8_to_nhwc_bf16_kernel(const uint8_t* __restrict__ x, int n, int ih, int iw, int oh, int ow,
                                              bf16* __restrict__ out, long long ld, float* __restrict__ out_nchw) {
  const long long total = static_cast<long long>(n) * oh * ow;
  const float sh = static_cast<float>(ih) / oh, sw = static_cast<float>(iw) / ow;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int ox = static_cast<int>(i % ow), oy = static_cast<int>((i / ow) % oh);
    const long long img = i / (static_cast<long long>(ow) * oh);
    const AaAxis ay = aa_axis(oy, ih, sh), ax = aa_axis(ox, iw, sw);
    float acc[C];
#pragma unroll
    for (int j = 0; j < C; ++j) acc[j] = 0.f;
    for (int jy = 0; jy < ay.n; ++jy) {
      const float wy = fmaxf(0.f, 1.f - fabsf((jy + ay.lo - ay.center + 0.5f) * ay.inv)) / ay.total;
      const uint8_t* row = x + ((img * ih + ay.lo + jy) * iw + ax.lo) * C;
      float r[C];
#pragma unroll
      for (int j = 0; j < C; ++j) r[j] = 0.f;
      for (int jx = 0; jx < ax.n; ++jx) {
        const float wx = fmaxf(0.f, 1.f - fabsf((jx + ax.lo - ax.center + 0.5f) * ax.inv)) / ax.total;
#pragma unroll
        for (int j = 0; j < C; ++j) r[j] = fmaf(wx, row[jx * C + j], r[j]);
      }
#pragma unroll
      for (int j = 0; j < C; ++j) acc[j] = fmaf(wy, r[j], acc[j]);
    }
    float v[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int j = 0; j < C; ++j) v[j] = acc[j] * (2.f / 255.f) - 1.f;
    if (out != nullptr) *reinterpret_cast<uint2*>(out + i * ld) = make_uint2(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]));
    if (out_nchw != nullptr) {      // what the reference's DataLoader yields: fp32 [n][C][oh][ow]
      const long long hw = static_cast<long long>(oh) * ow, pix = static_cast<long long>(oy) * ow + ox;
#pragma unroll
      for (int j = 0; j < C; ++j) out_nchw[(img * C + j) * hw + pix] = v[j];
    }
  }
}

// JointResize of the label map (dataset.py:143-146): NEAREST on the int64 {0,1} tensor, src = min(floor(dst*scale), in-1)
__global__ void resize_nearest_i64_kernel(const long long* __restrict__ x, int n, int ih, int iw, int oh, int ow,
                                          long long* __restrict__ out) {
  const long long total = static_cast<long long>(n) * oh * ow;
  const float sh = static_cast<float>(ih) / oh, sw = static_cast<float>(iw) / ow;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int ox = static_cast<int>(i % ow), oy = static_cast<int>((i / ow) % oh);
    const long long img = i / (static_cast<long long>(ow) * oh);
    const int sy = min(static_cast<int>(floorf(oy * sh)), ih - 1), sx = min(static_cast<int>(floorf(ox * sw)), iw - 1);
    out[i] = x[(img * ih + sy) * iw + sx];
  }
}

__global__ void sum_f32_kernel(const float* __restrict__ x, long long count, float* __restrict__ out) {
  float part = 0.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < count;
       i += (long long)gridDim.x * blockDim.x)
    part += x[i];
  part = warp_sum(part);
  __shared__ float red[32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) red[wid] = part;
  __syncthreads();
  if (wid == 0) {
    float v = lane < (blockDim.x >> 5) ? red[lane] : 0.f;
    v = warp_sum(v);
    if (lane == 0) atomicAdd(out, v);
  }
}

}  // namespace gap

using namespace gap;

// The streaming Cout = 1 kernels (cout1_z2 / cout1_wgrad2) cover c <= 512, 32-bit pixel indices and slopes for which
// LeakyReLU(v) = max(v, slope*v); `cout1_stream=0` (bring-up knob) forces the general kernels.
static bool cout1_streaming_ok(long long npix, int c, const float* in_scale, float in_slope) {
  if (debug_get("cout1_stream", 1) == 0) return false;
  if (c > 512 || npix > 0x7fffffe0LL) return false;
  if (in_scale && !(in_slope >= 0.f && in_slope <= 1.f)) return false;
  return true;
}

extern "C" {

int gap_cout1_conv_fwd(const void* x, int64_t ld_x, int n, int ih, int iw, int c, const void* w, const float* bias,
                       int ksize, int pad, float* z_ws, float* logits, const float* in_scale, const float* in_shift,
                       float in_slope, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  GAP_CHECK_ARG(x && w && z_ws && logits && n > 0 && ih > 0 && iw > 0, "gap_cout1_conv_fwd: bad arguments");
  GAP_CHECK_ARG((in_scale == nullptr) == (in_shift == nullptr) && (!in_scale || c <= 512),
                "gap_cout1_conv_fwd: in_scale / in_shift come together and need c <= 512");
  if (ksize != 4 || c % 64 != 0 || c <= 0 || ld_x % 8 != 0 || (reinterpret_cast<uintptr_t>(x) & 15) ||
      (reinterpret_cast<uintptr_t>(w) & 15)) {
    set_error("gap_cout1_conv_fwd: needs ksize 4, channels %% 64 == 0 and 16-byte aligned rows (c=%d ld=%lld)", c,
              (long long)ld_x);
    return GAP_ERR_UNSUPPORTED;
  }
  const int oh = ih + 2 * pad - 3, ow = iw + 2 * pad - 3;
  GAP_CHECK_ARG(oh > 0 && ow > 0, "gap_cout1_conv_fwd: empty output");
  const long long npix = static_cast<long long>(n) * ih * iw;
  const int tiles = static_cast<int>((npix + 127) / 128);
  const Cout1Pre pre{in_scale, in_shift, in_slope};
  if (cout1_streaming_ok(npix, c, in_scale, in_slope)) {
    // streaming kernel: one CTA per SM over 32-pixel tiles
    constexpr int smem = 128 + 8 * kC1Ring * kC1Unit + 2 * 8 * 256 * 4;
    static bool attr_set = false;
    if (!attr_set) {
      GAP_CUDA(cudaFuncSetAttribute(cout1_z2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
      GAP_CUDA(cudaFuncSetAttribute(cout1_z2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
      attr_set = true;
    }
    const int tiles32 = static_cast<int>((npix + 31) / 32);
    const int grid = std::min(tiles32, sm_count());
    if (in_scale)
      cout1_z2_kernel<true><<<grid, 256, smem, st>>>(static_cast<const bf16*>(x), ld_x, static_cast<int>(npix), c,
                                                      static_cast<const bf16*>(w), z_ws, pre);
    else
      cout1_z2_kernel<false><<<grid, 256, smem, st>>>(static_cast<const bf16*>(x), ld_x, static_cast<int>(npix), c,
                                                       static_cast<const bf16*>(w), z_ws, pre);
  } else if (in_scale) {
    cout1_z_kernel<true><<<std::min(tiles, 8 * sm_count()), 256, 0, st>>>(static_cast<const bf16*>(x), ld_x, npix, c,
                                                                           static_cast<const bf16*>(w), z_ws, pre);
  } else {
    cout1_z_kernel<false><<<std::min(tiles, 8 * sm_count()), 256, 0, st>>>(static_cast<const bf16*>(x), ld_x, npix, c,
                                                                            static_cast<const bf16*>(w), z_ws, pre);
  }
  GAP_CUDA(cudaGetLastError());
  const long long total = static_cast<long long>(n) * oh * ow;
  const int blocks = static_cast<int>(std::min<long long>((total + 63) / 64, 8LL * sm_count()));
  cout1_gather_kernel<<<blocks, 256, 0, st>>>(z_ws, bias, n, ih, iw, oh, ow, pad, logits);
  GAP_CUDA(cudaGetLastError());
  return 0;
}

static int cout1_dgrad_launch(const char* who, const float* dlogits, int n, int oh, int ow, const void* w, int ksize,
                              int pad, int c, void* gx, int64_t ld_gx, int ih, int iw, const Cout1Bwd* bwd, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!(dlogits && w && gx && n > 0 && oh > 0 && ow > 0 && ih > 0 && iw > 0)) {
    set_error("%s: bad arguments", who);
    return GAP_ERR_BAD_ARG;
  }
  if (ksize != 4 || c % 64 != 0 || c <= 0 || ld_gx % 8 != 0 || (reinterpret_cast<uintptr_t>(gx) & 15) ||
      (reinterpret_cast<uintptr_t>(w) & 15)) {
    set_error("%s: needs ksize 4, channels %% 64 == 0 and 16-byte aligned rows / weights", who);
    return GAP_ERR_UNSUPPORTED;
  }
  const long long npix = static_cast<long long>(n) * ih * iw;
  const size_t smem = (static_cast<size_t>(c) * 24 + 128 * 24 + 8 * 16 * 72) * sizeof(bf16) +
                      (bwd ? 128 + 8 * kC1YRing * kC1Unit : 0);
  if (smem > 200 * 1024) {
    set_error("%s: %d channels do not fit shared memory", who, c);
    return GAP_ERR_UNSUPPORTED;
  }
  static size_t attr[2] = {0, 0};
  const int v = bwd ? 1 : 0;
  if (smem > attr[v]) {
    if (bwd)
      GAP_CUDA(cudaFuncSetAttribute(cout1_dgrad_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    else
      GAP_CUDA(cudaFuncSetAttribute(cout1_dgrad_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    attr[v] = smem;
  }
  const int tiles = static_cast<int>((npix + 127) / 128);
  const int grid = std::min(tiles, 2 * sm_count());
  if (bwd)
    cout1_dgrad_kernel<true><<<grid, 256, smem, st>>>(dlogits, ih, iw, oh, ow, pad, npix, static_cast<const bf16*>(w), c,
                                                       static_cast<bf16*>(gx), ld_gx, *bwd);
  else
    cout1_dgrad_kernel<false><<<grid, 256, smem, st>>>(dlogits, ih, iw, oh, ow, pad, npix, static_cast<const bf16*>(w), c,
                                                        static_cast<bf16*>(gx), ld_gx, Cout1Bwd{});
  GAP_CUDA(cudaGetLastError());
  return 0;
}

int gap_cout1_conv_dgrad(const float* dlogits, int n, int oh, int ow, const void* w, int ksize, int pad, int c, void* gx,
                         int64_t ld_gx, int ih, int iw, void* stream) {
  return cout1_dgrad_launch("gap_cout1_conv_dgrad", dlogits, n, oh, ow, w, ksize, pad, c, gx, ld_gx, ih, iw, nullptr, stream);
}

int gap_cout1_conv_dgrad_bwd(const float* dlogits, int n, int oh, int ow, const void* w, int ksize, int pad, int c, void* gx,
                             int64_t ld_gx, int ih, int iw, const void* y, int64_t ld_y, const float* scale,
                             const float* shift, float slope, double* sums, void* stream) {
  GAP_CHECK_ARG(y && scale && shift && sums && c <= 512 && ld_y % 8 == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0,
                "gap_cout1_conv_dgrad_bwd: needs y / scale / shift / sums, c <= 512 and 16-byte aligned y rows");
  const Cout1Bwd b{static_cast<const bf16*>(y), ld_y, scale, shift, slope, sums};
  return cout1_dgrad_launch("gap_cout1_conv_dgrad_bwd", dlogits, n, oh, ow, w, ksize, pad, c, gx, ld_gx, ih, iw, &b, stream);
}

int gap_cout1_conv_wgrad(const float* dlogits, int n, int oh, int ow, const void* x, int64_t ld_x, int ih, int iw, int c,
                         int ksize, int pad, float* dw, const float* in_scale, const float* in_shift, float in_slope,
                         void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  GAP_CHECK_ARG(dlogits && x && dw && n > 0 && oh > 0 && ow > 0 && ih > 0 && iw > 0, "gap_cout1_conv_wgrad: bad arguments");
  GAP_CHECK_ARG((in_scale == nullptr) == (in_shift == nullptr), "gap_cout1_conv_wgrad: in_scale / in_shift come together");
  GAP_CHECK_ARG(!in_scale || 256 % (c / 8) == 0, "gap_cout1_conv_wgrad: the fused input transform needs c in {64, 128, 256, 512}");
  if (ksize != 4 || c % 64 != 0 || c <= 0 || c > 512 || ld_x % 8 != 0 || (reinterpret_cast<uintptr_t>(x) & 15)) {
    set_error("gap_cout1_conv_wgrad: needs ksize 4, channels %% 64 == 0, <= 512, 16-byte aligned rows");
    return GAP_ERR_UNSUPPORTED;
  }
  const long long npix = static_cast<long long>(n) * ih * iw;
  if (cout1_streaming_ok(npix, c, in_scale, in_slope)) {
    // streaming kernel: one CTA per SM, each a contiguous range of 16-pixel slabs
    constexpr int smem2 = 128 + 8 * kC1Ring * kC1Unit + kC1Round * 16 * 24 * 2;
    static bool attr_set = false;
    if (!attr_set) {
      GAP_CUDA(cudaFuncSetAttribute(cout1_wgrad2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem2));
      GAP_CUDA(cudaFuncSetAttribute(cout1_wgrad2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem2));
      attr_set = true;
    }
    const long long slabs = (npix + 15) / 16;
    // at most kC1Round slabs per CTA (one table round; larger inputs simply take more CTAs than SMs)
    const int per_cta = static_cast<int>(std::min<long long>((slabs + sm_count() - 1) / sm_count(), kC1Round));
    const int chunk2 = per_cta * 16;
    const int grid2 = static_cast<int>((npix + chunk2 - 1) / chunk2);
    const Cout1Pre pre2{in_scale, in_shift, in_slope};
    if (in_scale)
      cout1_wgrad2_kernel<true><<<grid2, 256, smem2, st>>>(dlogits, ih, iw, oh, ow, pad, static_cast<int>(npix), chunk2,
                                                            static_cast<const bf16*>(x), ld_x, c, dw, pre2);
    else
      cout1_wgrad2_kernel<false><<<grid2, 256, smem2, st>>>(dlogits, ih, iw, oh, ow, pad, static_cast<int>(npix), chunk2,
                                                             static_cast<const bf16*>(x), ld_x, c, dw, pre2);
    GAP_CUDA(cudaGetLastError());
    return 0;
  }
  const size_t smem = (static_cast<size_t>(16) * (c + 8) + 16 * 24) * sizeof(bf16) + (in_scale ? 2 * c * sizeof(float) : 0);
  const int want = debug_get("cout1_wg_mult", 4) * sm_count();
  long long chunk = (npix + want - 1) / want;
  chunk = (chunk + 15) / 16 * 16;
  const int grid = static_cast<int>((npix + chunk - 1) / chunk);
  const Cout1Pre pre{in_scale, in_shift, in_slope};
  if (in_scale)
    cout1_wgrad_kernel<true><<<grid, 256, smem, st>>>(dlogits, ih, iw, oh, ow, pad, npix, chunk,
                                                       static_cast<const bf16*>(x), ld_x, c, dw, pre);
  else
    cout1_wgrad_kernel<false><<<grid, 256, smem, st>>>(dlogits, ih, iw, oh, ow, pad, npix, chunk,
                                                        static_cast<const bf16*>(x), ld_x, c, dw, pre);
  GAP_CUDA(cudaGetLastError());
  return 0;
}

int gap_bce_logits_const_f32(const float* logits, int64_t count, float target, float grad_scale, float* dlogits,
                             double* loss_acc, float* dbias, void* stream) {
  GAP_CHECK_ARG(logits && loss_acc && count > 0, "gap_bce_logits_const_f32: bad arguments");
  const int blocks = static_cast<int>(std::min<int64_t>((count + 255) / 256, 148));
  bce_logits_const_f32_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(logits, count, target, grad_scale,
                                                                                     dlogits, loss_acc, dbias);
  GAP_CUDA(cudaGetLastError());
  return 0;
}

int gap_thin_conv_fwd(const void* src0, int64_t ld0, const void* src1, int64_t ld1, int n, int h, int w, const void* wpk,
                      const float* bias, int cw, void* out1, int64_t ldo1, int act1, void* out2, int64_t ldo2, int act2,
                      void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  GAP_CHECK_ARG(src0 && wpk && out1 && n > 0 && h > 1 && w > 1, "gap_thin_conv_fwd: bad arguments");
  GAP_CHECK_ARG(act1 >= GAP_ACT_NONE && act1 <= GAP_ACT_RELU && act2 >= GAP_ACT_NONE && act2 <= GAP_ACT_RELU,
                "gap_thin_conv_fwd: activations must be none / LeakyReLU / ReLU");
  if ((cw != 64 && cw != 128) || h % 2 || w % 2 || ld0 % 4 || (src1 && ld1 % 4) || ldo1 % 8 || (out2 && ldo2 % 8) ||
      (reinterpret_cast<uintptr_t>(src0) & 7) || (reinterpret_cast<uintptr_t>(src1) & 7) ||
      (reinterpret_cast<uintptr_t>(out1) & 15) || (reinterpret_cast<uintptr_t>(out2) & 15) ||
      (reinterpret_cast<uintptr_t>(wpk) & 15)) {
    set_error("gap_thin_conv_fwd: needs cw in {64,128}, even h/w, 4-slot sources (ld %% 4), 16-byte aligned outputs");
    return GAP_ERR_UNSUPPORTED;
  }
  ThinFwdParams p;
  p.s0 = static_cast<const bf16*>(src0);
  p.ld0 = ld0;
  p.s1 = static_cast<const bf16*>(src1);
  p.ld1 = ld1;
  p.w = static_cast<const bf16*>(wpk);
  p.bias = bias;
  p.n = n;
  p.h = h;
  p.w_in = w;
  p.oh = h / 2;
  p.ow = w / 2;
  p.cw = cw;
  auto slope_of = [](int act) { return act == GAP_ACT_NONE ? 1.f : (act == GAP_ACT_LRELU ? 0.2f : 0.f); };
  p.out1 = static_cast<bf16*>(out1);
  p.ldo1 = ldo1;
  p.slope1 = slope_of(act1);
  p.out2 = static_cast<bf16*>(out2);
  p.ldo2 = ldo2;
  p.slope2 = slope_of(act2);
  p.tiles_x = (p.ow + 15) / 16;
  p.tiles_y = (p.oh + 7) / 8;
  p.total_tiles = static_cast<long long>(n) * p.tiles_x * p.tiles_y;
  GAP_CHECK_ARG(p.total_tiles < (1ll << 31), "gap_thin_conv_fwd: too many tiles");
  p.skip = debug_get("thin_skip", 0);
  const int ct = src1 ? 8 : 4;
  for (int o = 0; o < 2; ++o) {
    const void* base = o == 0 ? out1 : out2;
    const int64_t ldo = o == 0 ? ldo1 : ldo2;
    if (base == nullptr) continue;
    const uint64_t ld_b = static_cast<uint64_t>(ldo) * 2;
    uint64_t dims[4] = {static_cast<uint64_t>(cw), static_cast<uint64_t>(p.ow), static_cast<uint64_t>(p.oh),
                        static_cast<uint64_t>(n)};
    uint64_t strides[3] = {ld_b, ld_b * p.ow, ld_b * p.ow * p.oh};
    uint32_t box[4] = {64, 16, 8, 1};
    int rc = encode_tmap_bf16(&p.tm_out[o], base, 4, dims, strides, box, nullptr, true);
    if (rc) return rc;
    if (p.ow == 128) {
      uint32_t box_row[4] = {64, 128, 1, 1};
      rc = encode_tmap_bf16(&p.tm_row[o], base, 4, dims, strides, box_row, nullptr, true);
      if (rc) return rc;
    }
  }
  // full-width dense rows: the tcgen05 row kernel (see thin_conv_fwd_tc_kernel)
  const bool tc_ok = w == 256 && ld0 == 4 && (!src1 || ld1 == 4) && ldo1 % 16 == 0 && (!out2 || ldo2 % 16 == 0) &&
                     (reinterpret_cast<uintptr_t>(out1) & 31) == 0 && (reinterpret_cast<uintptr_t>(out2) & 31) == 0 &&
                     (!bias || (reinterpret_cast<uintptr_t>(bias) & 15) == 0) && !(cw == 128 && out2) &&
                     debug_get("thin_tc", 1) != 0;
  if (tc_ok) {
    const int kc = 16 * ct / 8;
    const size_t smem_tc = 1024 + static_cast<size_t>(2) * (out2 ? 2 : 1) * (cw / 64) * 16384 + static_cast<size_t>(kc) * cw * 16 +
                           kTcSlots * 2 * (ct == 8 ? 2 : 1) * kTcPlane + (2 * kTcSlots + 8) * 8 + 16;
    const int grid_tc = std::min(n * p.oh, 2 * sm_count());
    static bool set_tc = false;
    if (!set_tc) {
      GAP_CUDA(cudaFuncSetAttribute(thin_conv_fwd_tc_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024));
      GAP_CUDA(cudaFuncSetAttribute(thin_conv_fwd_tc_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024));
      set_tc = true;
    }
    if (ct == 8)
      thin_conv_fwd_tc_kernel<8><<<grid_tc, kTcThreads, smem_tc, st>>>(p);
    else
      thin_conv_fwd_tc_kernel<4><<<grid_tc, kTcThreads, smem_tc, st>>>(p);
    GAP_CUDA(cudaGetLastError());
    return 0;
  }
  const size_t smem = 1024 + static_cast<size_t>(cw / 64) * 16384 + 2 * 18 * 34 * ct * 2 +
                      static_cast<size_t>(cw) * (16 * ct + 8) * 2;
  const int threads = 128 * (cw / 64);
  const int grid = static_cast<int>(std::min<long long>(p.total_tiles, static_cast<long long>(debug_get("thin_ctas_per_sm", 4)) * sm_count()));
  if (ct == 8) {
    static bool set8 = false;
    if (!set8) {
      GAP_CUDA(cudaFuncSetAttribute(thin_conv_fwd_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
      set8 = true;
    }
    thin_conv_fwd_kernel<8><<<grid, threads, smem, st>>>(p);
  } else {
    static bool set4 = false;
    if (!set4) {
      GAP_CUDA(cudaFuncSetAttribute(thin_conv_fwd_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
      set4 = true;
    }
    thin_conv_fwd_kernel<4><<<grid, threads, smem, st>>>(p);
  }
  GAP_CUDA(cudaGetLastError());
  return 0;
}

static int thin_conv_wgrad_launch(const void* wide, int64_t ld_w, const void* src0, int64_t ld0, const void* src1,
                                  int64_t ld1, int c0, int c1, int n, int h, int w, int cw, float* dw, int64_t ld_m,
                                  float* dbias, void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if ((cw != 64 && cw != 128) || h % 2 || w % 2 || ld0 % 4 || (src1 && ld1 % 4) || ld_w % 8 ||
      (reinterpret_cast<uintptr_t>(src0) & 7) || (reinterpret_cast<uintptr_t>(src1) & 7) ||
      (reinterpret_cast<uintptr_t>(wide) & 15)) {
    set_error("gap_thin_conv_wgrad: needs cw in {64,128}, even h/w, 4-slot sources (ld %% 4), 16-byte aligned wide rows");
    return GAP_ERR_UNSUPPORTED;
  }
  ThinWgradParams p;
  p.wide = static_cast<const bf16*>(wide);
  p.ld_w = ld_w;
  p.s0 = static_cast<const bf16*>(src0);
  p.ld0 = ld0;
  p.s1 = static_cast<const bf16*>(src1);
  p.ld1 = ld1;
  p.n = n;
  p.h = h;
  p.w_in = w;
  p.oh = h / 2;
  p.ow = w / 2;
  p.cw = cw;
  p.dw = dw;
  p.ld_m = ld_m;
  p.c0 = c0;
  p.c1 = c1;
  p.c_real = c0 + c1;
  p.dbias = dbias;
  p.tiles_x = (p.ow + 15) / 16;
  p.tiles_y = (p.oh + 7) / 8;
  p.total_tiles = static_cast<long long>(n) * p.tiles_x * p.tiles_y;
  GAP_CHECK_ARG(p.total_tiles < (1ll << 31), "gap_thin_conv_wgrad: too many tiles");
  const int ct = src1 ? 8 : 4;
  {
    const uint64_t ld_b = static_cast<uint64_t>(ld_w) * 2;
    uint64_t dims[4] = {static_cast<uint64_t>(cw), static_cast<uint64_t>(p.ow), static_cast<uint64_t>(p.oh),
                        static_cast<uint64_t>(n)};
    uint64_t strides[3] = {ld_b, ld_b * p.ow, ld_b * p.ow * p.oh};
    uint32_t box[4] = {64, 16, 8, 1};
    int rc = encode_tmap_bf16(&p.tm_wide, wide, 4, dims, strides, box, nullptr, true);
    if (rc) return rc;
  }
  // full-width dense rows: the tcgen05 row kernel (see thin_conv_wgrad_tc_kernel)
  if (w == 256 && ld0 == 4 && (!src1 || ld1 == 4) && debug_get("thin_tc", 1) != 0) {
    const uint64_t ld_b = static_cast<uint64_t>(ld_w) * 2;
    uint64_t dims[4] = {static_cast<uint64_t>(cw), static_cast<uint64_t>(p.ow), static_cast<uint64_t>(p.oh),
                        static_cast<uint64_t>(n)};
    uint64_t strides[3] = {ld_b, ld_b * p.ow, ld_b * p.ow * p.oh};
    uint32_t box_row[4] = {64, 128, 1, 1};
    int rc = encode_tmap_bf16(&p.tm_row, wide, 4, dims, strides, box_row, nullptr, true);
    if (rc) return rc;
    const size_t smem_tc = 1024 + 4 * static_cast<size_t>(cw / 64) * 16384 + 8 * 2 * (ct == 8 ? 4 : 2) * 2048 + 32 * 8 +
                           2 * 16 * 64 * 4;
    const int grid_tc = std::min(n * p.oh, sm_count());
    static bool set_tc = false;
    if (!set_tc) {
      GAP_CUDA(cudaFuncSetAttribute(thin_conv_wgrad_tc_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
      GAP_CUDA(cudaFuncSetAttribute(thin_conv_wgrad_tc_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
      set_tc = true;
    }
    if (ct == 8)
      thin_conv_wgrad_tc_kernel<8><<<grid_tc, kWtThreads, smem_tc, st>>>(p);
    else
      thin_conv_wgrad_tc_kernel<4><<<grid_tc, kWtThreads, smem_tc, st>>>(p);
    GAP_CUDA(cudaGetLastError());
    return 0;
  }
  const size_t smem = 1024 + 2 * static_cast<size_t>(cw / 64) * 16384 + 2 * 18 * 34 * ct * 2 + 16;
  const int threads = 128 * (cw / 64);
  const int grid = static_cast<int>(std::min<long long>(p.total_tiles, static_cast<long long>(debug_get("thin_wgrad_ctas_per_sm", 3)) * sm_count()));
  if (ct == 8) {
    static bool set8 = false;
    if (!set8) {
      GAP_CUDA(cudaFuncSetAttribute(thin_conv_wgrad_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
      set8 = true;
    }
    thin_conv_wgrad_kernel<8><<<grid, threads, smem, st>>>(p);
  } else {
    static bool set4 = false;
    if (!set4) {
      GAP_CUDA(cudaFuncSetAttribute(thin_conv_wgrad_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
      set4 = true;
    }
    thin_conv_wgrad_kernel<4><<<grid, threads, smem, st>>>(p);
  }
  GAP_CUDA(cudaGetLastError());
  return 0;
}

int gap_thin_conv_wgrad(const void* wide, int64_t ld_w, const void* src0, int64_t ld0, const void* src1, int64_t ld1,
                        int n, int h, int w, int cw, float* dw, int64_t ld_m, float* dbias, void* stream) {
  GAP_CHECK_ARG(wide && src0 && dw && n > 0 && h > 1 && w > 1, "gap_thin_conv_wgrad: bad arguments");
  return thin_conv_wgrad_launch(wide, ld_w, src0, ld0, src1, ld1, 3, src1 ? 3 : 0, n, h, w, cw, dw, ld_m, dbias, stream);
}

int gap_thin_conv_wgrad_c(const void* wide, int64_t ld_w, const void* src0, int64_t ld0, int c0, const void* src1,
                          int64_t ld1, int c1, int n, int h, int w, int cw, float* dw, int64_t ld_m, float* dbias,
                          void* stream) {
  GAP_CHECK_ARG(c0 >= 1 && c0 <= 4 && (src1 ? (c1 >= 1 && c1 <= 4) : c1 == 0),
                "gap_thin_conv_wgrad_c: c0 must be 1..4, c1 1..4 with a second source and 0 without");
  GAP_CHECK_ARG(wide && src0 && dw && n > 0 && h > 1 && w > 1, "gap_thin_conv_wgrad_c: bad arguments");
  return thin_conv_wgrad_launch(wide, ld_w, src0, ld0, src1, ld1, c0, c1, n, h, w, cw, dw, ld_m, dbias, stream);
}

}  // extern "C"

template <int CO>
static int thin_convT_launch(const void* wide, int64_t ld_w, int n, int ih, int iw, int cw, const void* wcol, const float* bias,
                             int act, void* out_bf16, int64_t ld_bf, float* out_f32, int64_t ld_f, uint8_t* out_u8,
                             void* stream) {
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  GAP_CHECK_ARG(act == GAP_ACT_NONE || act == GAP_ACT_TANH, "gap_thin_convT_fwd: activation must be none or Tanh");
  if ((cw != 64 && cw != 128) || ld_w % 8 || (out_bf16 && ld_bf % 4) || (out_f32 && ld_f % 4) ||
      (reinterpret_cast<uintptr_t>(wide) & 15) || (reinterpret_cast<uintptr_t>(wcol) & 15) ||
      (reinterpret_cast<uintptr_t>(out_bf16) & 7) || (reinterpret_cast<uintptr_t>(out_f32) & 15)) {
    set_error("gap_thin_convT_fwd: needs cw in {64,128}, 16-byte aligned wide rows and 4-slot outputs");
    return GAP_ERR_UNSUPPORTED;
  }
  ThinConvTParams p;
  p.wide = static_cast<const bf16*>(wide);
  p.ld_w = ld_w;
  p.wcol = static_cast<const bf16*>(wcol);
  p.bias = bias;
  p.n = n;
  p.ih = ih;
  p.iw = iw;
  p.cw = cw;
  p.act = act;
  p.out_bf = static_cast<bf16*>(out_bf16);
  p.ld_bf = ld_bf;
  p.out_f32 = out_f32;
  p.ld_f = ld_f;
  p.out_u8 = out_u8;
  p.tiles_x = (iw + 15) / 16;
  p.tiles_y = (ih + 7) / 8;
  p.total_tiles = static_cast<long long>(n) * p.tiles_x * p.tiles_y;
  GAP_CHECK_ARG(p.total_tiles < (1ll << 31), "gap_thin_convT_fwd: too many tiles");
  {
    const uint64_t ld_b = static_cast<uint64_t>(ld_w) * 2;
    uint64_t dims[4] = {static_cast<uint64_t>(cw), static_cast<uint64_t>(iw), static_cast<uint64_t>(ih),
                        static_cast<uint64_t>(n)};
    uint64_t strides[3] = {ld_b, ld_b * iw, ld_b * iw * ih};
    uint32_t box[4] = {64, 18, 10, 1};
    int rc = encode_tmap_bf16(&p.tm_wide, wide, 4, dims, strides, box, nullptr, true);
    if (rc) return rc;
  }
  const size_t smem = 1024 + static_cast<size_t>(cw / 64) * kWideTileBytes + 16 * CO * static_cast<size_t>(cw + 8) * 2 +
                      192 * thin_convT_col_stride(CO) * 4 + 16;
  static bool set = false;
  if (!set) {
    GAP_CUDA(cudaFuncSetAttribute(thin_convT_fwd_kernel<CO>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    set = true;
  }
  const int grid = static_cast<int>(std::min<long long>(p.total_tiles, static_cast<long long>(debug_get("thin_convT_ctas_per_sm", cw == 64 ? 3 : 2)) * sm_count()));
  thin_convT_fwd_kernel<CO><<<grid, 256, smem, st>>>(p);
  GAP_CUDA(cudaGetLastError());
  return 0;
}

extern "C" {

int gap_thin_convT_fwd(const void* wide, int64_t ld_w, int n, int ih, int iw, int cw, const void* wcol, const float* bias,
                       int act, void* out_bf16, int64_t ld_bf, float* out_f32, int64_t ld_f, uint8_t* out_u8, void* stream) {
  GAP_CHECK_ARG(wide && wcol && (out_bf16 || out_f32 || out_u8) && n > 0 && ih > 0 && iw > 0, "gap_thin_convT_fwd: bad arguments");
  return thin_convT_launch<3>(wide, ld_w, n, ih, iw, cw, wcol, bias, act, out_bf16, ld_bf, out_f32, ld_f, out_u8, stream);
}

int gap_thin_convT_fwd_c(const void* wide, int64_t ld_w, int n, int ih, int iw, int cw, int co, const void* wcol,
                         const float* bias, int act, void* out_bf16, int64_t ld_bf, float* out_f32, int64_t ld_f,
                         uint8_t* out_u8, void* stream) {
  GAP_CHECK_ARG(co >= 1 && co <= 4, "gap_thin_convT_fwd_c: co must be 1..4");
  GAP_CHECK_ARG(wide && wcol && (out_bf16 || out_f32 || out_u8) && n > 0 && ih > 0 && iw > 0, "gap_thin_convT_fwd_c: bad arguments");
  switch (co) {
    case 1: return thin_convT_launch<1>(wide, ld_w, n, ih, iw, cw, wcol, bias, act, out_bf16, ld_bf, out_f32, ld_f, out_u8, stream);
    case 2: return thin_convT_launch<2>(wide, ld_w, n, ih, iw, cw, wcol, bias, act, out_bf16, ld_bf, out_f32, ld_f, out_u8, stream);
    case 3: return thin_convT_launch<3>(wide, ld_w, n, ih, iw, cw, wcol, bias, act, out_bf16, ld_bf, out_f32, ld_f, out_u8, stream);
    default: return thin_convT_launch<4>(wide, ld_w, n, ih, iw, cw, wcol, bias, act, out_bf16, ld_bf, out_f32, ld_f, out_u8, stream);
  }
}

int gap_u8_hwc_to_nhwc_bf16(const uint8_t* x, void* out, int64_t out_ld, int64_t pixels, void* stream) {
  return gap_u8_hwc_to_nhwc_bf16_c(x, 3, out, out_ld, pixels, stream);
}

int gap_u8_hwc_to_nhwc_bf16_c(const uint8_t* x, int c, void* out, int64_t out_ld, int64_t pixels, void* stream) {
  GAP_CHECK_ARG(c >= 1 && c <= 4, "gap_u8_hwc_to_nhwc_bf16_c: c must be 1..4");
  GAP_CHECK_ARG(x && out && pixels > 0 && out_ld % 4 == 0 && (reinterpret_cast<uintptr_t>(out) & 7) == 0,
                "gap_u8_hwc_to_nhwc_bf16: bad arguments");
  const int blocks = static_cast<int>(std::min<int64_t>((pixels + 255) / 256, 148 * 16));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  bf16* o = static_cast<bf16*>(out);
  switch (c) {
    case 1: u8_hwc_to_nhwc_bf16_kernel<1><<<blocks, 256, 0, st>>>(x, o, out_ld, pixels); break;
    case 2: u8_hwc_to_nhwc_bf16_kernel<2><<<blocks, 256, 0, st>>>(x, o, out_ld, pixels); break;
    case 3: u8_hwc_to_nhwc_bf16_kernel<3><<<blocks, 256, 0, st>>>(x, o, out_ld, pixels); break;
    default: u8_hwc_to_nhwc_bf16_kernel<4><<<blocks, 256, 0, st>>>(x, o, out_ld, pixels); break;
  }
  GAP_CUDA(cudaGetLastError());
  return 0;
}

int gap_resize_u8_to_nhwc_bf16(const uint8_t* x, int n, int ih, int iw, int oh, int ow, void* out, int64_t out_ld,
                               float* out_nchw_f32, void* stream) {
  return gap_resize_u8_to_nhwc_bf16_c(x, 3, n, ih, iw, oh, ow, out, out_ld, out_nchw_f32, stream);
}

int gap_resize_u8_to_nhwc_bf16_c(const uint8_t* x, int c, int n, int ih, int iw, int oh, int ow, void* out, int64_t out_ld,
                                 float* out_nchw_f32, void* stream) {
  GAP_CHECK_ARG(c >= 1 && c <= 4, "gap_resize_u8_to_nhwc_bf16_c: c must be 1..4");
  GAP_CHECK_ARG(x && (out || out_nchw_f32) && n > 0 && ih > 0 && iw > 0 && oh > 0 && ow > 0 &&
                    (!out || (out_ld >= 4 && out_ld % 4 == 0)),
                "gap_resize_u8_to_nhwc_bf16: bad arguments");
  const long long total = static_cast<long long>(n) * oh * ow;
  const int blocks = static_cast<int>(std::min<long long>((total + 255) / 256, 148 * 16));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  bf16* o = static_cast<bf16*>(out);
  switch (c) {
    case 1: resize_u8_to_nhwc_bf16_kernel<1><<<blocks, 256, 0, st>>>(x, n, ih, iw, oh, ow, o, out_ld, out_nchw_f32); break;
    case 2: resize_u8_to_nhwc_bf16_kernel<2><<<blocks, 256, 0, st>>>(x, n, ih, iw, oh, ow, o, out_ld, out_nchw_f32); break;
    case 3: resize_u8_to_nhwc_bf16_kernel<3><<<blocks, 256, 0, st>>>(x, n, ih, iw, oh, ow, o, out_ld, out_nchw_f32); break;
    default: resize_u8_to_nhwc_bf16_kernel<4><<<blocks, 256, 0, st>>>(x, n, ih, iw, oh, ow, o, out_ld, out_nchw_f32); break;
  }
  GAP_CUDA(cudaGetLastError());
  return 0;
}

int gap_resize_nearest_i64(const int64_t* x, int n, int ih, int iw, int oh, int ow, int64_t* out, void* stream) {
  GAP_CHECK_ARG(x && out && n > 0 && ih > 0 && iw > 0 && oh > 0 && ow > 0, "gap_resize_nearest_i64: bad arguments");
  const long long total = static_cast<long long>(n) * oh * ow;
  const int blocks = static_cast<int>(std::min<long long>((total + 255) / 256, 148 * 16));
  resize_nearest_i64_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const long long*>(x), n, ih, iw, oh, ow, reinterpret_cast<long long*>(out));
  GAP_CUDA(cudaGetLastError());
  return 0;
}

int gap_sum_f32(const float* x, int64_t count, float* out, void* stream) {
  GAP_CHECK_ARG(x && out && count > 0, "gap_sum_f32: bad arguments");
  const int blocks = static_cast<int>(std::min<int64_t>((count + 255) / 256, 148));
  sum_f32_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(x, count, out);
  GAP_CUDA(cudaGetLastError());
  return 0;
}

}  // extern "C"
